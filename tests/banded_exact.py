"""Exact banded alignment: orc_align_banded (tests/banded_oracle.c) restated in Python integers.  TEST INFRASTRUCTURE ONLY.

The band, borders, recurrence, end cell, predecessor order and local 0-floor stop are those of orc_fill_banded and
orc_traceback_full with start and end type -1, in both modes.  Only the band's cells are stored.  There are no int32
lanes and no saturation: every finite value is exact however far below -2^31 it falls, and -infinity is
float("-inf").  The record reports -infinity as po.NEG (the ABI's PSA_NEG_INF) and every finite value as it is, so a
value that the int32 oracle saturates, or that a kernel cuts off as "no path", shows up as a difference.

The rule the banded entries apply to (g, h) in global mode (csrc/psa_capi.cu, check_banded_scoring) is mirrored below.
"""
from __future__ import annotations

from oracle.pyoracle import GLOBAL, LOCAL, NEG, Alignment

NEG_INF = float("-inf")
SPAN_LIMIT = 1 << 28


# ---- the range rule of the banded entries ----------------------------------------------------------------------

def span(g, h, m, n):
    """check_scoring's span (three gap openings): the full matrix, local mode, and band >= max(m, n)."""
    return g * (m + n + 2) + 2 * h + m + n


def span_banded(g, h, m, n):
    """check_banded_scoring's span for a global call with band < max(m, n): one opening per gap run of an optimal path."""
    return g * (m + n + 2) + h * (min(m, n) + 3) + m + n


def largest_h(m, n, g, rule=span_banded):
    return (SPAN_LIMIT - 1 - rule(g, 0, m, n)) // (rule(g, 1, m, n) - rule(g, 0, m, n))


def largest_g(m, n, h, rule=span_banded):
    return (SPAN_LIMIT - 1 - rule(0, h, m, n)) // (m + n + 2)


# ---- fill and traceback ----------------------------------------------------------------------------------------

def band_rows(m, n, band):
    """(lo, hi) of rows 0 .. m: the columns |j - floor(i*n/m)| <= band.  With m = 0 or n = 0 every cell (the band plays
    no role there, as in orc_align_banded)."""
    if m == 0 or n == 0:
        return [(0, n)] * (m + 1)
    return [(max(0, i * n // m - band), min(n, i * n // m + band)) for i in range(m + 1)]


class BandedTables:
    """T1, T2, T3 on the band's cells: row i holds columns rows[i][0] .. rows[i][1]."""

    def __init__(self, a: bytes, b: bytes, band: int, g: int, h: int, mode: int):
        m, n = len(a), len(b)
        self.rows = rows = band_rows(m, n, band)
        go = g + h
        glob = mode == GLOBAL
        hi0 = rows[0][1]
        T1 = [[0 if glob else NEG_INF] + [NEG_INF] * hi0]
        T2 = [[NEG_INF] + [-h - g * j if glob else NEG_INF for j in range(1, hi0 + 1)]]
        T3 = [[NEG_INF] * (hi0 + 1)]
        for i in range(1, m + 1):
            lo, hi = rows[i]
            plo, phi = rows[i - 1]
            p1, p2, p3 = T1[-1], T2[-1], T3[-1]
            r1, r2, r3 = [], [], []
            ai = a[i - 1]
            for j in range(lo, hi + 1):
                if j == 0:
                    r1.append(NEG_INF)
                    r2.append(NEG_INF)
                    r3.append(-h - g * i if glob else NEG_INF)
                    continue
                x = j - 1 - plo                        # (i-1, j-1) in the row above, then (i-1, j)
                d = max(p1[x], p2[x], p3[x]) if plo <= j - 1 <= phi else NEG_INF
                if not glob:
                    d = max(d, 0)
                r1.append(d + (1 if ai == b[j - 1] else 0))
                r3.append(max(p1[x + 1] - go, p2[x + 1] - go, p3[x + 1] - g) if plo <= j <= phi else NEG_INF)
                r2.append(max(r1[-2] - go, r2[-1] - g, r3[-2] - go) if j > lo else NEG_INF)
            T1.append(r1)
            T2.append(r2)
            T3.append(r3)
        self.T = (None, T1, T2, T3)

    def get(self, t, i, j):
        lo, hi = self.rows[i]
        return self.T[t][i][j - lo] if lo <= j <= hi else NEG_INF


def _abi(v):
    return NEG if v == NEG_INF else v


def render_rows(a, b, ops, start_i, start_j):
    """orc_render_rows: the two printed rows of forward ops starting at cell (start_i, start_j)."""
    ra, rb = bytearray(), bytearray()
    i, j = start_i, start_j
    for k, t in enumerate(ops):
        if k:
            i += t != 2
            j += t != 3
        ra.append(a[i - 1] if t in (1, 3) else 0x2D)
        rb.append(b[j - 1] if t in (1, 2) else 0x2D)
    return bytes(ra), bytes(rb)


def align_banded(a: bytes, b: bytes, band: int, g: int = 1, h: int = 2, mode: int = GLOBAL) -> Alignment:
    """bo.align_banded in exact arithmetic: record, ops (forward, 1/2/3), rows, and the no-path record of a global
    call whose band admits no path from (0, 0) to (m, n)."""
    m, n = len(a), len(b)
    tab = BandedTables(a, b, band, g, h, mode)
    go = g + h
    if mode == GLOBAL:
        t1, t2, t3 = (tab.get(t, m, n) for t in (1, 2, 3))
        if max(t1, t2, t3) == NEG_INF:
            return Alignment(NEG, NEG, NEG, NEG, 1, m, n, 0, 0, b"", b"", b"")
        state = 1 if (t1 >= t2 and t1 >= t3) else (2 if (t2 >= t1 and t2 >= t3) else 3)
        score, i, j = max(t1, t2, t3), m, n
    else:
        best, i, j = 0, 0, 0
        for r in range(1, m + 1):
            lo, hi = tab.rows[r]
            for c in range(max(lo, 1), hi + 1):
                if tab.get(1, r, c) > best:
                    best, i, j = tab.get(1, r, c), r, c
        t1, t2, t3, score, state = best, NEG_INF, NEG_INF, best, 1
    end = (i, j)
    end_state = state
    ops = []
    si = sj = 0
    while i > 0 and j > 0:
        ops.append(state)
        si, sj = i, j
        f = 1 if a[i - 1] == b[j - 1] else 0
        if state == 1:
            v = tab.get(1, i, j)
            if mode == LOCAL and v == f:             # the 0-floor first: this is the first column
                break
            prev = [tab.get(t, i - 1, j - 1) + f for t in (1, 2, 3)]
            i, j = i - 1, j - 1
        elif state == 2:
            v = tab.get(2, i, j)
            prev = [tab.get(1, i, j - 1) - go, tab.get(2, i, j - 1) - g, tab.get(3, i, j - 1) - go]
            j -= 1
        else:
            v = tab.get(3, i, j)
            prev = [tab.get(1, i - 1, j) - go, tab.get(2, i - 1, j) - go, tab.get(3, i - 1, j) - g]
            i -= 1
        assert v in prev, ("no predecessor", i, j, state)
        state = prev.index(v) + 1
    ops = bytes(reversed(ops))
    ra, rb = render_rows(a, b, ops, si, sj)
    return Alignment(_abi(t1), _abi(t2), _abi(t3), _abi(score), end_state, end[0], end[1], si, sj, ops, ra, rb)
