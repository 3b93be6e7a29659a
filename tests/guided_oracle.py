"""ctypes doorway to tests/guided_oracle.c, the CPU restatement of psa_align_batch_guided (TEST INFRASTRUCTURE ONLY),
and guide_rows, the band of an anchor chain restated from include/psa.h.

The library is compiled on first use into a temporary directory named after the hash of its sources, so that the
repository tree is never written to."""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
import threading

import numpy as np

from oracle.pyoracle import GLOBAL, Alignment, OrcResult

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = [os.path.join(HERE, "guided_oracle.c"), os.path.join(HERE, "banded_oracle.c"),
           os.path.join(HERE, "..", "oracle", "gotoh_oracle.c")]

_lib = None


def _build() -> str:
    h = hashlib.sha256()
    for p in SOURCES:
        with open(p, "rb") as f:
            h.update(f.read())
    out_dir = os.path.join(tempfile.gettempdir(), f"psa_guided_oracle_{h.hexdigest()[:16]}")
    so = os.path.join(out_dir, "libguided_oracle.so")
    if not os.path.exists(so):
        os.makedirs(out_dir, exist_ok=True)
        tmp = f"{so}.{os.getpid()}.{threading.get_ident()}"      # unique per thread: concurrent first uses each build
        subprocess.check_call([os.environ.get("CC", "cc"), "-O2", "-Wall", "-shared", "-fPIC", "-o", tmp, SOURCES[0]])
        os.replace(tmp, so)
    return so


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(_build())
        _lib.orc_align_rows.restype = C.c_int
        _lib.orc_align_rows.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                        C.c_void_p, C.POINTER(OrcResult), C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.orc_score_rows.restype = C.c_int
        _lib.orc_score_rows.argtypes = [C.c_char_p, C.c_char_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                        C.c_void_p, C.POINTER(OrcResult)]
    return _lib


def diag_rows(m: int, n: int, band: int):
    """(lo, hi) of the diagonal band, |j - floor(i*n/m)| <= band, as orc_band_lo / orc_band_hi compute them."""
    c = np.arange(m + 1, dtype=np.int64) * n // m
    return np.maximum(0, c - band), np.minimum(n, c + band)


def guide_rows(m: int, n: int, anchors, band: int):
    """(lo, hi) int64 arrays over rows 0 .. m of the band around an anchor chain, restated from include/psa.h: the guide
    is the polyline (0, 0), P_1 .. P_K, (m, n); a row with chain points on it spans the j of its first and last point,
    any other row takes floor of the segment crossing it; lo = max(0, cmin - band), hi = min(n, cmax + band).  Raises
    ValueError for an invalid chain (a coordinate outside [0, m] x [0, n] or decreasing along the chain).  With m = 0 or
    n = 0 every cell (the band plays no role there)."""
    P = np.asarray(anchors, dtype=np.int64).reshape(-1, 2)
    if len(P) and (P[:, 0].min() < 0 or P[:, 0].max() > m or P[:, 1].min() < 0 or P[:, 1].max() > n):
        raise ValueError("anchor outside the matrix")
    if len(P) > 1 and (np.diff(P[:, 0]).min() < 0 or np.diff(P[:, 1]).min() < 0):
        raise ValueError("anchor chain decreases")
    if m == 0 or n == 0:
        return np.zeros(m + 1, np.int64), np.full(m + 1, n, np.int64)
    P = np.concatenate([[[0, 0]], P, [[m, n]]])
    cmin = np.full(m + 1, np.iinfo(np.int64).max)
    cmax = np.full(m + 1, -1)
    for (i0, j0), (i1, j1) in zip(P[:-1], P[1:]):
        if i1 > i0 + 1:                       # rows strictly inside the segment
            r = np.arange(i0 + 1, i1)
            c = j0 + (r - i0) * (j1 - j0) // (i1 - i0)
            cmin[r] = c
            cmax[r] = c
    for i, j in P:                            # chain points: first and last on their row (j is non-decreasing)
        cmin[i] = min(cmin[i], j)
        cmax[i] = max(cmax[i], j)
    return np.maximum(0, cmin - band), np.minimum(n, cmax + band)


def align_rows(a: bytes, b: bytes, lo, hi, g: int = 1, h: int = 2, mode: int = GLOBAL) -> Alignment:
    """Full-table oracle over per-row bands lo[i] <= j <= hi[i]: fill + traceback + rows."""
    m, n = len(a), len(b)
    lo = np.ascontiguousarray(lo, dtype=np.int64)
    hi = np.ascontiguousarray(hi, dtype=np.int64)
    res = OrcResult()
    ops = np.zeros(m + n + 1, dtype=np.uint8)
    ra = np.zeros(m + n + 1, dtype=np.uint8)
    rb = np.zeros(m + n + 1, dtype=np.uint8)
    rc = lib().orc_align_rows(a, b, m, n, g, h, mode, lo.ctypes.data, hi.ctypes.data, C.byref(res), ops.ctypes.data,
                              ra.ctypes.data, rb.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"orc_align_rows rc={rc}")
    L = res.aln_len
    return Alignment(res.t1, res.t2, res.t3, res.score, res.end_state, res.end_i, res.end_j, res.start_i,
                     res.start_j, ops[:L].tobytes(), ra[:L].tobytes(), rb[:L].tobytes())


def score_rows(a: bytes, b: bytes, lo, hi, g: int = 1, h: int = 2, mode: int = GLOBAL) -> OrcResult:
    """Linear-space score and end cell over per-row bands."""
    lo = np.ascontiguousarray(lo, dtype=np.int64)
    hi = np.ascontiguousarray(hi, dtype=np.int64)
    res = OrcResult()
    rc = lib().orc_score_rows(a, b, len(a), len(b), g, h, mode, lo.ctypes.data, hi.ctypes.data, C.byref(res))
    if rc != 0:
        raise RuntimeError(f"orc_score_rows rc={rc}")
    return res
