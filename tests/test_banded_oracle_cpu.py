"""The banded restatement in tests/banded_oracle.c (orc_align_banded, orc_score_banded) against the unbanded oracle:
a band that holds every cell changes nothing, a narrower band can only lose score, and the linear-space form agrees
with the full-table form.  No GPU."""
import random

import numpy as np
import pytest

from oracle import pyoracle as po
from tests import banded_oracle as bo
from tests.helpers import mutated_copy, py_random_pair, random_dna

GRID = [(1, 2), (0, 0), (0, 1), (2, 0), (3, 1), (5, 2)]


def _same(x, y):
    return (x.t1, x.t2, x.t3, x.score, x.end_state, x.end_i, x.end_j, x.start_i, x.start_j, x.ops, x.row_a, x.row_b) == \
           (y.t1, y.t2, y.t3, y.score, y.end_state, y.end_i, y.end_j, y.start_i, y.start_j, y.ops, y.row_a, y.row_b)


@pytest.mark.parametrize("mode", [po.GLOBAL, po.LOCAL])
@pytest.mark.parametrize("g,h", GRID)
def test_wide_band_is_the_full_oracle(mode, g, h):
    rnd = random.Random(4100 + 10 * g + h + 100 * mode)
    for _ in range(60):
        a, b = py_random_pair(rnd, 40, 48)
        full = po.align(a, b, g, h, mode=mode)
        for band in (max(len(a), len(b)), max(len(a), len(b)) + 7):
            assert _same(bo.align_banded(a, b, band, g, h, mode), full), (a, b, band)
            lin = bo.score_banded(a, b, band, g, h, mode)
            assert (lin.score, lin.end_i, lin.end_j) == (full.score, full.end_i, full.end_j)


@pytest.mark.parametrize("mode", [po.GLOBAL, po.LOCAL])
def test_score_monotone_in_band_and_linear_form_agrees(mode):
    rng = np.random.default_rng(4200 + mode)
    rnd = random.Random(4201 + mode)
    pairs = [py_random_pair(rnd, 60, 60) for _ in range(20)]
    for _ in range(10):
        a = random_dna(rng, int(rng.integers(50, 120)))
        pairs.append((a, mutated_copy(rng, a, int(rng.integers(40, 140)))))
    for a, b in pairs:
        full = po.align(a, b, mode=mode)
        prev = None
        for band in (0, 1, 2, 3, 5, 8, 13, 21, 40, 200):
            got = bo.align_banded(a, b, band, mode=mode)
            lin = bo.score_banded(a, b, band, mode=mode)
            assert (lin.t1, lin.t2, lin.t3, lin.score, lin.end_state, lin.end_i, lin.end_j) == \
                   (got.t1, got.t2, got.t3, got.score, got.end_state, got.end_i, got.end_j), (a, b, band)
            assert got.score <= full.score
            if prev is not None:
                assert got.score >= prev
            prev = got.score
            if got.score > po.NEG and got.ops:
                # every cell of the reported alignment lies inside the band
                m, n = len(a), len(b)
                i, j = got.start_i, got.start_j
                for k, t in enumerate(got.ops):
                    if k:
                        i += t != 2
                        j += t != 3
                    assert abs(j - i * n // m) <= band, (a, b, band, i, j)


def test_no_global_path_reports_minus_infinity():
    a = b"A"
    b = b"ACGT" * 250
    got = bo.align_banded(a, b, 10)
    assert (got.t1, got.t2, got.t3, got.score, got.end_state, got.end_i, got.end_j, got.ops) == \
           (po.NEG, po.NEG, po.NEG, po.NEG, 1, 1, 1000, b"")
    lin = bo.score_banded(a, b, 10)
    assert (lin.t1, lin.score, lin.end_state, lin.aln_len) == (po.NEG, po.NEG, 1, 0)
    # local mode always has a (possibly empty) answer
    loc = bo.align_banded(a, b, 10, mode=po.LOCAL)
    assert loc.score == 1 and loc.end_i == 1


def test_empty_members_are_the_full_oracle():
    for a, b in ((b"", b"ACG"), (b"ACG", b""), (b"", b"")):
        for mode in (po.GLOBAL, po.LOCAL):
            assert _same(bo.align_banded(a, b, 0, mode=mode), po.align(a, b, mode=mode))
