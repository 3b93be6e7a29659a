"""Shared test helpers: FASTA fixture reader and seeded sequence generators (SURVEY 8d)."""
import hashlib
import os
import random

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def read_fasta(path):
    names, seqs, cur = [], [], []
    with open(path) as f:
        for line in f:
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


_dataset = None


def dataset():
    global _dataset
    if _dataset is None:
        _dataset = read_fasta(os.path.join(GOLDEN, "dataset_head.fa"))
    return _dataset


def random_dna(rng: np.random.Generator, n: int) -> bytes:
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, size=n)].tobytes()


def mutated_copy(rng: np.random.Generator, a: bytes, n: int, sub=0.05, ins=0.01, dele=0.01) -> bytes:
    """B = mutated copy of A: substitutions, short geometric insertions/deletions, pad/trim to n."""
    alpha = b"ACGT"
    out = bytearray()
    i = 0
    while i < len(a):
        r = rng.random()
        if r < dele:
            i += int(rng.geometric(0.5))
            continue
        if r < dele + ins:
            for _ in range(int(rng.geometric(0.5))):
                out.append(alpha[int(rng.integers(0, 4))])
        c = a[i]
        if rng.random() < sub:
            c = alpha[(alpha.index(c) + int(rng.integers(1, 4))) % 4] if c in alpha else alpha[0]
        out.append(c)
        i += 1
    while len(out) < n:
        out.append(alpha[int(rng.integers(0, 4))])
    return bytes(out[:n])


def py_random_pair(rnd: random.Random, max_m=40, max_n=48, alpha=b"ACGT"):
    m = rnd.randint(1, max_m)
    n = rnd.randint(m, max(m, max_n))
    a = bytes(rnd.choice(alpha) for _ in range(m))
    if rnd.random() < 0.5:
        bb = bytearray(a)
        for k in range(len(bb)):
            if rnd.random() < 0.12:
                bb[k] = rnd.choice(alpha)
        while len(bb) < n:
            bb.insert(rnd.randint(0, len(bb)), rnd.choice(alpha))
        b = bytes(bb)
    else:
        b = bytes(rnd.choice(alpha) for _ in range(n))
    return a, b


def table_record(tables, corner, end_state, ops: bytes, row_a: bytes, row_b: bytes):
    """What the full-table comparisons check, small enough to store: tables [3, m+1, n+1] int32 (-inf = NEG)."""
    return {"tables_md5": [hashlib.md5(t.astype("<i4").tobytes()).hexdigest() for t in tables],
            "corner": [int(x) for x in corner], "end_state": int(end_state), "ops": "".join(str(x) for x in ops),
            "rows_md5": hashlib.md5(row_a + b"\n" + row_b + b"\n").hexdigest()}
