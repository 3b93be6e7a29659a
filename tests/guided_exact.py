"""Exact alignment over per-row bands: orc_align_rows (tests/guided_oracle.c) restated in Python integers.  TEST
INFRASTRUCTURE ONLY.

The per-row twin of tests/banded_exact.py: the same borders, recurrence, end cell, predecessor order and local 0-floor
stop, with row i's cells lo(i) <= j <= hi(i) given as `rows` (the band of an anchor chain, guided_oracle.guide_rows)
instead of the diagonal band.  No int32 lanes, no saturation: -infinity is float("-inf") and is reported as po.NEG.
"""
from __future__ import annotations

from oracle.pyoracle import GLOBAL, LOCAL, NEG, Alignment
from tests.banded_exact import NEG_INF, render_rows


class RowTables:
    """T1, T2, T3 on the band's cells: row i holds columns rows[i][0] .. rows[i][1]."""

    def __init__(self, a: bytes, b: bytes, rows, g: int, h: int, mode: int):
        m = len(a)
        self.rows = rows
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
                x = j - 1 - plo
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


def align_rows(a: bytes, b: bytes, rows, g: int = 1, h: int = 2, mode: int = GLOBAL) -> Alignment:
    """go.align_rows in exact arithmetic: record, forward ops, rows, and the no-path record of a global call
    whose band admits no path from (0, 0) to (m, n)."""
    m, n = len(a), len(b)
    tab = RowTables(a, b, rows, g, h, mode)
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
            lo, hi = rows[r]
            for c in range(max(lo, 1), hi + 1):
                if tab.get(1, r, c) > best:
                    best, i, j = tab.get(1, r, c), r, c
        t1, t2, t3, score, state = best, NEG_INF, NEG_INF, best, 1
    end, end_state = (i, j), state
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
