"""ctypes doorway to tests/banded_oracle.c, the CPU restatement of psa_align_batch_banded (TEST INFRASTRUCTURE ONLY).

The library is compiled on first use into a temporary directory named after the hash of its sources, so that the
repository tree is never written to."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle.pyoracle import GLOBAL, Alignment, OrcResult

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "banded_oracle.c"), os.path.join(HERE, "..", "oracle", "gotoh_oracle.c")]

_lib = None


def _build() -> str:
    h = hashlib.sha256()
    for p in SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"psa_banded_oracle_{h.hexdigest()[:16]}")
    so = os.path.join(out_dir, "libbanded_oracle.so")
    if not os.path.exists(so):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{so}.{os.getpid()}"
        subprocess.check_call([os.environ.get("CC", "cc"), "-O2", "-Wall", "-shared", "-fPIC", "-o", tmp, SOURCES[0]])
        os.replace(tmp, so)
    return so


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(_build())
        _lib.orc_align_banded.restype = C.c_int
        _lib.orc_align_banded.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int,
                                          C.c_int64, C.POINTER(OrcResult), C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.orc_score_banded.restype = C.c_int
        _lib.orc_score_banded.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int,
                                          C.c_int64, C.POINTER(OrcResult)]
    return _lib


def align_banded(a: bytes, b: bytes, band: int, g: int = 1, h: int = 2, mode: int = GLOBAL) -> Alignment:
    """Full-table banded oracle (cells with |j - floor(i*n/m)| > band are -inf): fill + traceback + rows."""
    m, n = len(a), len(b)
    res = OrcResult()
    ops = np.zeros(m + n + 1, dtype=np.uint8)
    ra = np.zeros(m + n + 1, dtype=np.uint8)
    rb = np.zeros(m + n + 1, dtype=np.uint8)
    rc = lib().orc_align_banded(a, b, m, n, g, h, mode, band, C.byref(res), ops.ctypes.data, ra.ctypes.data,
                                rb.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orc_align_banded rc={rc}")
    L = res.aln_len
    return Alignment(res.t1, res.t2, res.t3, res.score, res.end_state, res.end_i, res.end_j, res.start_i,
                     res.start_j, ops[:L].tobytes(), ra[:L].tobytes(), rb[:L].tobytes())


def score_banded(a: bytes, b: bytes, band: int, g: int = 1, h: int = 2, mode: int = GLOBAL) -> OrcResult:
    """Linear-space banded score and end cell (O(band) memory per row)."""
    res = OrcResult()
    rc = lib().orc_score_banded(a, b, len(a), len(b), g, h, mode, band, C.byref(res))
    if rc != 0:
        raise RuntimeError(f"orc_score_banded rc={rc}")
    return res
