"""The oracle (oracle/gotoh_oracle.c) against the reference's golden vectors (SURVEY 8c), against the full-table
answers stored in tests/golden/ref_tables.json and, where the compiled reference is built (oracle/_ref), against the
reference itself on the same seeded pairs.  CPU only."""
import hashlib
import json
import os
import random

import numpy as np

from oracle import pyoracle as po
from tests.helpers import GOLDEN, dataset, py_random_pair, table_record


def _check(case, a, b):
    al = po.align(a, b, case["g"], case["h"])
    assert [al.t1, al.t2, al.t3] == case["corner"]
    assert al.end_state == case["end_state"]
    assert len(al.ops) == case["cols"]
    assert (al.ops.count(1), al.ops.count(2), al.ops.count(3)) == (case["n_t1"], case["n_t2"], case["n_t3"])
    assert hashlib.md5(al.row_a + b"\n" + al.row_b + b"\n").hexdigest() == case["md5"]
    if "row_a" in case:
        assert al.row_a.decode() == case["row_a"] and al.row_b.decode() == case["row_b"]
    lin = po.score_linear(a, b, case["g"], case["h"])
    assert [lin.t1, lin.t2, lin.t3] == case["corner"]


def test_kat_vectors():
    names, seqs = dataset()
    for case in json.load(open(os.path.join(GOLDEN, "kat.json"))):
        if "a" in case:
            a, b = case["a"].encode(), case["b"].encode()
        else:
            if case["L"] > 3000:
                continue  # long ones: test_kat_long
            a, b = seqs[case["rec_a"]][:case["L"]].encode(), seqs[case["rec_b"]][:case["L"]].encode()
        _check(case, a, b)


def test_kat_long():
    names, seqs = dataset()
    for case in json.load(open(os.path.join(GOLDEN, "kat.json"))):
        if case.get("L", 0) > 3000:
            a, b = seqs[case["rec_a"]][:case["L"]].encode(), seqs[case["rec_b"]][:case["L"]].encode()
            _check(case, a, b)


def test_random_small_fixture():
    for case in json.load(open(os.path.join(GOLDEN, "random_small.json"))):
        _check(case, case["a"].encode(), case["b"].encode())


def test_typed_subproblem_fixture():
    """Every (start_type, end_type) border variant of Subproblem, answers recorded from the reference
    (tests/golden/make_golden.py::typed_fixture)."""
    cases = json.load(open(os.path.join(GOLDEN, "typed_small.json")))
    assert len({(c["start_type"], c["end_type"]) for c in cases}) == 36
    for case in cases:
        al = po.align(case["a"].encode(), case["b"].encode(), case["g"], case["h"], start_type=case["start_type"],
                      end_type=case["end_type"])
        assert [al.t1, al.t2, al.t3] == case["corner"] and al.end_state == case["end_state"]
        assert al.row_a.decode() == case["row_a"] and al.row_b.decode() == case["row_b"]


def test_g1_pair_is_config1():
    """BASELINE config 1: records #2 and #15, first 50 bp, rows as printed by the reference."""
    names, seqs = dataset()
    lines = open(os.path.join(GOLDEN, "g1_stdout.txt")).read().split("\n")
    al = po.align(seqs[2][:50].encode(), seqs[15][:50].encode(), 1, 2)
    assert al.row_a.decode() in lines and al.row_b.decode() in lines
    assert (al.t1, al.t2, al.t3, al.end_state) == (9, 5, 7, 1)


def _stored_tables():
    return json.load(open(os.path.join(GOLDEN, "ref_tables.json")))


def test_oracle_equals_reference_random():
    """Full T1/T2/T3 tables, corner, end state, node states and printed rows of 400 seeded pairs against the answers
    stored in ref_tables.json and, where oracle/_ref is built, against the live reference on the same inputs."""
    for case in _stored_tables()["random"]:
        a, b, g, h = case["a"].encode(), case["b"].encode(), case["g"], case["h"]
        al, T = po.align(a, b, g, h, want_tables=True)
        got = table_record(T, (al.t1, al.t2, al.t3), al.end_state, al.ops, al.row_a, al.row_b)
        assert all(got[k] == case[k] for k in got), (case, got)
        if po.have_ref():
            corner, es, nodes, RT = po.ref_subproblem(a, b, g, h, p=case["p"], want_tables=True)
            assert np.array_equal(T, RT)
            assert (al.t1, al.t2, al.t3) == tuple(int(x) for x in corner) and al.end_state == es
            ra, rb = po.ref_rows(a, b, nodes)
            assert (al.row_a, al.row_b) == (ra, rb)
            assert al.ops == bytes(nodes[:, 2].astype(np.uint8))


def test_oracle_equals_reference_typed_tables():
    """Full T1/T2/T3 tables, end state and node states for all 36 (start, end) types against the answers stored in
    ref_tables.json and, where oracle/_ref is built, against the live reference on the same inputs."""
    cases = _stored_tables()["typed"]
    assert len({(c["start_type"], c["end_type"]) for c in cases}) == 36
    for case in cases:
        a, b, g, h = case["a"].encode(), case["b"].encode(), case["g"], case["h"]
        st, et = case["start_type"], case["end_type"]
        al, T = po.align(a, b, g, h, start_type=st, end_type=et, want_tables=True)
        got = table_record(T, (al.t1, al.t2, al.t3), al.end_state, al.ops, al.row_a, al.row_b)
        assert all(got[k] == case[k] for k in got if k != "rows_md5"), (case, got)
        if po.have_ref():
            c, es, nodes, RT = po.ref_subproblem(a, b, g, h, p=case["p"], start_type=st, end_type=et, want_tables=True)
            assert np.array_equal(T, RT) and al.end_state == es
            assert al.ops == bytes(nodes[:, 2].astype(np.uint8))


# main_alignment_function(AGGA, AGTGC, p=3, g=1, h=2) as the reference prints it: its breadcrumbs, then print_seq's rows
REFERENCE_STDOUT_AGGA = b"bp1\nbp1.2\nbp2\nbp3\nbp4\nAG-GA\nAGTGC\n"


def test_reference_stdout_format():
    """The reference's printed answer for AGGA x AGTGC: its rows are the oracle's rows; where oracle/_ref is built,
    the live reference still prints exactly these bytes."""
    al = po.align(b"AGGA", b"AGTGC", 1, 2)
    assert REFERENCE_STDOUT_AGGA.split(b"\n")[5:7] == [al.row_a, al.row_b]
    if po.have_ref():
        assert po.ref_main_alignment_stdout(b"AGGA", b"AGTGC", 3, 1, 2) == REFERENCE_STDOUT_AGGA


def test_local_mode_properties():
    """Local mode has no reference: check the spec's invariants on random pairs."""
    rnd = random.Random(11)
    for t in range(300):
        a, b = py_random_pair(rnd)
        g, h = rnd.choice([(1, 2), (2, 1), (1, 0)])
        al, T = po.align(a, b, g, h, mode=po.LOCAL, want_tables=True)
        lin = po.score_linear(a, b, g, h, mode=po.LOCAL)
        assert (lin.score, lin.end_i, lin.end_j) == (al.score, al.end_i, al.end_j)
        assert al.score == max(0, int(T[0][1:, 1:].max()))
        if al.score == 0:
            assert al.ops == b""
            continue
        # rows re-score to the reported score; first/last columns are matches
        s, gap = 0, 0
        for x, y in zip(al.row_a, al.row_b):
            if x == 0x2D or y == 0x2D:
                kind = 2 if x == 0x2D else 3
                s -= g + (h if gap != kind else 0)
                gap = kind
            else:
                s += 1 if x == y else 0
                gap = 0
        assert s == al.score
        assert al.ops[0] == 1 and al.ops[-1] == 1 and al.row_a[0] == al.row_b[0]
        assert al.row_a.replace(b"-", b"") == a[al.start_i - 1:al.end_i]
        assert al.row_b.replace(b"-", b"") == b[al.start_j - 1:al.end_j]
