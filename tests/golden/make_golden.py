"""Regenerates the golden fixtures in this directory FROM THE REFERENCE ITSELF.

Runs only in the build container (needs /root/reference and oracle/_ref built by
`make -C oracle ref`).  The outputs are committed; nothing at test time reads /root/reference.

  dataset_head.fa   the 20 FASTA records of gene_sequences_test, each truncated to HEAD bases
                    (enough for every golden prefix below); 70-column lines like the original
  g1_stdout.txt     full stdout of the reference program (BASELINE config 1; SURVEY 8c "G1")
  kat.json          known-answer vectors: corner values, end state, printed rows (or their
                    md5 + op counts for long ones) as produced by the reference's Subproblem
  random_small.json 400 seeded random/mutated pairs with the reference's full answers
  typed_small.json  the 36 (start_type, end_type) border variants of Subproblem, 8 pairs each
  ref_tables.json   the inputs of tests/test_oracle_golden.py's two full-table comparisons, each with an md5 of
                    T1, T2 and T3, the corner, the end state, the node states and (random pairs) an md5 of the printed rows;
                    taken from the reference when oracle/_ref is built, else from the oracle, and the file's
                    "source" says which (ref_tables_fixture, which can run on its own)

Usage:  python tests/golden/make_golden.py [tables]
"""
import hashlib
import json
import os
import random
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import pyoracle as po  # noqa: E402
from tests.helpers import py_random_pair, table_record  # noqa: E402

REF_DATA = "/root/reference/gene_sequences_test"
HEAD = 13400


def read_fasta(path):
    names, seqs, cur = [], [], []
    for line in open(path):
        line = line.rstrip("\n")
        if line.startswith(">"):
            if cur:
                seqs.append("".join(cur))
                cur = []
            names.append(line)
        else:
            cur.append(line)
    if cur:
        seqs.append("".join(cur))
    return names, seqs


def ref_case(a: bytes, b: bytes, g, h, p=1, keep_rows=True, start_type=-1, end_type=-1):
    corner, end_state, nodes = po.ref_subproblem(a, b, g, h, p=p, start_type=start_type, end_type=end_type)
    ra, rb = po.ref_rows(a, b, nodes)
    t = nodes[:, 2] if len(nodes) else []
    out = {
        "g": g, "h": h, "m": len(a), "n": len(b),
        "corner": [int(x) for x in corner], "end_state": int(end_state), "cols": int(len(nodes)),
        "n_t1": int(sum(1 for x in t if x == 1)), "n_t2": int(sum(1 for x in t if x == 2)),
        "n_t3": int(sum(1 for x in t if x == 3)),
        "md5": hashlib.md5(ra + b"\n" + rb + b"\n").hexdigest(),
    }
    if keep_rows:
        out["row_a"] = ra.decode()
        out["row_b"] = rb.decode()
    return out


def main():
    po.build()
    names, seqs = read_fasta(REF_DATA)
    assert len(names) == 20 and len(seqs) == 20

    with open(os.path.join(HERE, "dataset_head.fa"), "w") as f:
        for nm, s in zip(names, seqs):
            f.write(nm + "\n")
            s = s[:HEAD]
            for k in range(0, len(s), 70):
                f.write(s[k:k + 70] + "\n")

    # G1: the reference program, shipped flags, run against the full data file
    with tempfile.TemporaryDirectory() as td:
        os.symlink(REF_DATA, os.path.join(td, "gene_sequences_test"))
        out = subprocess.run([os.path.join(ROOT, "oracle", "_ref", "testing_ref")], cwd=td, capture_output=True,
                             check=True).stdout.decode()
        csv = open(os.path.join(td, "input_size_testing.csv")).read()
    with open(os.path.join(HERE, "g1_stdout.txt"), "w") as f:
        f.write(out)
    with open(os.path.join(HERE, "g1_csv_head.txt"), "w") as f:
        f.write("\n".join(csv.split("\n")[:2]) + "\n")

    kat = []
    # G2..G5: the reference's own commented-out fragments + survey probes
    for name, a, b, g, h in [
        ("G2_main_alignment.cpp:356-362", b"AGGA", b"AGTGC", 1, 2),
        ("G3_subproblem_alignment.cpp:190-200", b"AGGA", b"ATGTC", 2, 1),
        ("G4", b"ACGTACGTAC", b"ACGTTACGAC", 1, 2),
        ("G5", b"ACGTACGTACGTACGTTTGACA", b"ACGTAACGTACGTACGTTTGACA", 1, 2),
    ]:
        c = ref_case(a, b, g, h, p=3)
        c.update(name=name, a=a.decode(), b=b.decode())
        kat.append(c)
    # G6: dataset prefixes (records r1, r2, prefix L of both)
    for r1, r2, L in [(2, 15, 50), (2, 15, 150), (2, 15, 1000), (2, 15, 10000), (0, 1, 10000), (6, 8, 13327),
                      (3, 11, 777), (19, 4, 2500)]:
        L = min(L, len(seqs[r1]), len(seqs[r2]))
        a, b = seqs[r1][:L].encode(), seqs[r2][:L].encode()
        c = ref_case(a, b, 1, 2, p=1, keep_rows=(L <= 1000))
        c.update(name=f"G6_dataset_{r1}_{r2}_{L}", rec_a=r1, rec_b=r2, L=L)
        kat.append(c)
    json.dump(kat, open(os.path.join(HERE, "kat.json"), "w"), indent=1)

    rnd = random.Random(20250001)
    cases = []
    for t in range(400):
        m = rnd.randint(1, 96)
        n = rnd.randint(m, min(128, m + rnd.choice([0, 0, 1, 3, 10, 40])))
        alpha = rnd.choice([b"ACGT", b"ACGT", b"AC", b"ACGTN", b"ABCDEFGHIJKLMNOPQRSTUVWY"])
        a = bytes(rnd.choice(alpha) for _ in range(m))
        if rnd.random() < 0.6:
            bb = bytearray(a)
            for k in range(len(bb)):
                if rnd.random() < 0.1:
                    bb[k] = rnd.choice(alpha)
            while len(bb) < n:
                bb.insert(rnd.randint(0, len(bb)), rnd.choice(alpha))
            b = bytes(bb)
        else:
            b = bytes(rnd.choice(alpha) for _ in range(n))
        g, h = rnd.choice([(1, 2), (1, 2), (1, 2), (2, 1), (1, 0), (0, 2), (3, 5), (1, 1), (0, 0)])
        c = ref_case(a, b, g, h, p=rnd.choice([1, 3, 32]))
        c.update(a=a.decode(), b=b.decode())
        cases.append(c)
    json.dump(cases, open(os.path.join(HERE, "random_small.json"), "w"))
    typed_fixture()
    ref_tables_fixture()
    print("golden fixtures written:", len(kat), "KATs,", len(cases), "random cases")


def typed_fixture():
    """Subproblem with every (start_type, end_type) in {-1,-2,-3,1,2,3}^2 (subproblem_alignment.cpp:
    212-227, 259-292, 112-146): what optimal_alignment (main_alignment.cpp:250-251) passes for the
    pieces of a partitioned alignment."""
    rnd = random.Random(20250002)
    cases = []
    for st in (-1, -2, -3, 1, 2, 3):
        for et in (-1, -2, -3, 1, 2, 3):
            for t in range(8):
                m = rnd.randint(1, 48)
                n = rnd.randint(m, m + rnd.choice([0, 1, 5, 20]))
                a = bytes(rnd.choice(b"ACGT") for _ in range(m))
                bb = bytearray(a if rnd.random() < 0.6 else bytes(rnd.choice(b"ACGT") for _ in range(m)))
                for k in range(len(bb)):
                    if rnd.random() < 0.15:
                        bb[k] = rnd.choice(b"ACGT")
                while len(bb) < n:
                    bb.insert(rnd.randint(0, len(bb)), rnd.choice(b"ACGT"))
                g, h = rnd.choice([(1, 2), (1, 2), (2, 1), (1, 0), (0, 2), (1, 1)])
                c = ref_case(a, bytes(bb), g, h, p=rnd.choice([1, 3]), start_type=st, end_type=et)
                c.update(a=a.decode(), b=bytes(bb).decode(), start_type=st, end_type=et)
                cases.append(c)
    json.dump(cases, open(os.path.join(HERE, "typed_small.json"), "w"))
    print("typed fixture written:", len(cases), "cases")


def _ref_record(a, b, g, h, p, start_type=-1, end_type=-1):
    if po.have_ref():
        corner, end_state, nodes, tables = po.ref_subproblem(a, b, g, h, p=p, start_type=start_type, end_type=end_type,
                                                             want_tables=True)
        ra, rb = po.ref_rows(a, b, nodes)
        return table_record(tables, corner, end_state, bytes(int(x) for x in nodes[:, 2]), ra, rb)
    al, tables = po.align(a, b, g, h, start_type=start_type, end_type=end_type, want_tables=True)
    return table_record(tables, (al.t1, al.t2, al.t3), al.end_state, al.ops, al.row_a, al.row_b)


def ref_tables_fixture():
    """The exact seeded draws of test_oracle_equals_reference_random (random.Random(7)) and
    test_oracle_equals_reference_typed_tables (random.Random(5)), with their answers."""
    out = {"source": "reference (oracle/_ref)" if po.have_ref() else
           "oracle (gotoh_oracle.c): the compiled reference was not available when this file was written",
           "random": [], "typed": []}
    rnd = random.Random(7)
    for t in range(400):
        a, b = py_random_pair(rnd, alpha=rnd.choice([b"ACGT", b"AC", b"ACGTN"]))
        g, h = rnd.choice([(1, 2), (1, 2), (2, 1), (1, 0), (0, 3), (4, 7), (0, 0)])
        p = rnd.choice([1, 2, 5, 32])
        out["random"].append(dict(a=a.decode(), b=b.decode(), g=g, h=h, p=p, **_ref_record(a, b, g, h, p)))
    rnd = random.Random(5)
    for st in (-1, -2, -3, 1, 2, 3):
        for et in (-1, -2, -3, 1, 2, 3):
            for t in range(6):
                m = rnd.randint(1, 30)
                n = rnd.randint(m, 36)
                a = bytes(rnd.choice(b"ACGT") for _ in range(m))
                b = bytes(rnd.choice(b"ACGT") for _ in range(n))
                g, h = rnd.choice([(1, 2), (2, 1), (1, 0), (0, 2)])
                p = rnd.choice([1, 3])
                rec = _ref_record(a, b, g, h, p, st, et)
                del rec["rows_md5"]                 # the typed comparison checks tables, end state and node states
                out["typed"].append(dict(a=a.decode(), b=b.decode(), g=g, h=h, p=p, start_type=st, end_type=et, **rec))
    json.dump(out, open(os.path.join(HERE, "ref_tables.json"), "w"), separators=(",", ":"))
    print("full-table fixture written:", len(out["random"]), "random,", len(out["typed"]), "typed cases;", out["source"])


if __name__ == "__main__":
    if sys.argv[1:] == ["tables"]:
        po.build()
        ref_tables_fixture()
    else:
        main()
