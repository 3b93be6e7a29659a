"""ctypes bindings of include/psa.h (libpsa.so).  No torch types cross the C boundary: device
entry points take raw pointers (tensor.data_ptr()) and a raw cudaStream_t."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Iterable, Optional, Sequence

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
GLOBAL, LOCAL = 0, 1
WANT_SCORE, WANT_TRACEBACK, OPS_COMPACT = 1, 2, 4
NEG_INF = -(2 ** 31) // 2


class PsaError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libpsa error {code}: {msg}")
        self.code = code


class BatchItem(C.Structure):
    _fields_ = [("t1", C.c_int32), ("t2", C.c_int32), ("t3", C.c_int32), ("score", C.c_int32),
                ("end_state", C.c_int32), ("end_i", C.c_int32), ("end_j", C.c_int32), ("start_i", C.c_int32),
                ("start_j", C.c_int32), ("aln_len", C.c_int32)]


BP_DTYPE = np.dtype([("i", "<i8"), ("j", "<i8"), ("t", "<i4"), ("reserved", "<i4")])   # psa_bp
ITEM_DTYPE = np.dtype([("t1", "<i4"), ("t2", "<i4"), ("t3", "<i4"), ("score", "<i4"), ("end_state", "<i4"),
                       ("end_i", "<i4"), ("end_j", "<i4"), ("start_i", "<i4"), ("start_j", "<i4"),
                       ("aln_len", "<i4")])
assert ITEM_DTYPE.itemsize == C.sizeof(BatchItem) == 40
PACKED_ITEM_DTYPE = np.dtype([("score", "<i4"), ("end_i", "<u2"), ("end_j", "<u2"), ("start_i", "<u2"), ("start_j", "<u2"),
                              ("aln_len", "<u2"), ("end_state", "<u2")])    # psa_packed_item
assert PACKED_ITEM_DTYPE.itemsize == 16


class _Result(C.Structure):
    _fields_ = [("t1", C.c_int32), ("t2", C.c_int32), ("t3", C.c_int32), ("score", C.c_int32),
                ("end_state", C.c_int32), ("end_i", C.c_int64), ("end_j", C.c_int64), ("start_i", C.c_int64),
                ("start_j", C.c_int64), ("aln_len", C.c_int64), ("ops", C.POINTER(C.c_uint8)),
                ("row_a", C.POINTER(C.c_char)), ("row_b", C.POINTER(C.c_char))]   # raw bytes: a sequence may contain NUL


def library_path() -> str:
    # PSA_LIBRARY: another build of the same ABI, for A/B timing of two kernel versions on one box (tools/ only)
    return os.environ.get("PSA_LIBRARY") or os.path.join(HERE, "libpsa.so")


def build_library(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libpsa.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(HERE, "csrc"), "-j8"]
    if not verbose:
        cmd.insert(1, "-s")
    subprocess.check_call(cmd)
    # the reference-shaped C++ program (host/testing) links against the library just built
    subprocess.check_call(["make", "-s", "-C", os.path.join(HERE, "host")])
    return library_path()


_lib: Optional[C.CDLL] = None


def load_library() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise PsaError(-3, f"{path} is missing: build it with __graft_entry__.build() "
                           "(there is no CPU fallback for the alignment kernels)")
    lib = C.CDLL(path)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    lib.psa_ctx_create.restype = C.c_int
    lib.psa_ctx_create.argtypes = [C.c_int, C.POINTER(vp)]
    lib.psa_ctx_destroy.restype = None
    lib.psa_ctx_destroy.argtypes = [vp]
    lib.psa_last_error.restype = C.c_char_p
    lib.psa_last_error.argtypes = [vp]
    lib.psa_launch_count.restype = i64
    lib.psa_launch_count.argtypes = [vp]
    lib.psa_ctx_set_option.restype = C.c_int          # csrc/psa_internal.h: test / measurement hook
    lib.psa_ctx_set_option.argtypes = [vp, C.c_char_p, C.c_longlong]
    lib.psa_align_pair.restype = C.c_int
    lib.psa_align_pair.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                   C.c_uint, C.POINTER(_Result)]
    lib.psa_align_pair_typed.restype = C.c_int
    lib.psa_align_pair_typed.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                         C.c_int, C.c_uint, C.POINTER(_Result)]
    lib.psa_similarity_batch.restype = C.c_int
    lib.psa_similarity_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_size_t, C.c_size_t, vp]
    lib.psa_similarity_batch_device.restype = C.c_int
    lib.psa_similarity_batch_device.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_int, vp, vp]
    lib.psa_align_partition.restype = C.c_int
    lib.psa_align_partition.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t, C.c_size_t, vp, C.c_size_t, C.c_int, C.c_int,
                                        C.POINTER(_Result)]
    lib.psa_align_long_partitioned.restype = C.c_int
    lib.psa_align_long_partitioned.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                               C.POINTER(_Result), vp, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.psa_result_free.restype = None
    lib.psa_result_free.argtypes = [C.POINTER(_Result)]
    lib.psa_align_batch.restype = C.c_int
    lib.psa_align_batch.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int,
                                    C.c_int, C.c_int, C.c_uint, vp, vp, C.c_size_t]
    lib.psa_pack_bases.restype = C.c_size_t
    lib.psa_pack_bases.argtypes = [vp, C.c_size_t, vp]
    lib.psa_pack_reads.restype = C.c_size_t
    lib.psa_pack_reads.argtypes = [vp, C.c_size_t, C.c_size_t, C.c_size_t, vp, C.c_int]
    lib.psa_align_batch_packed.restype = C.c_int
    lib.psa_align_batch_packed.argtypes = [vp, vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint, vp, vp,
                                           C.c_size_t]
    lib.psa_align_batch_device.restype = C.c_int
    lib.psa_align_batch_device.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                           C.c_int, C.c_int, C.c_uint, vp, vp, C.c_size_t, vp]
    lib.psa_align_batch_banded.restype = C.c_int
    lib.psa_align_batch_banded.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int,
                                           C.c_int, C.c_int, C.c_int, C.c_uint, vp, vp, C.c_size_t]
    lib.psa_align_batch_banded_device.restype = C.c_int
    lib.psa_align_batch_banded_device.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_int, C.c_int, C.c_int,
                                                  C.c_int, C.c_int, C.c_int, C.c_uint, vp, vp, C.c_size_t, vp]
    lib.psa_align_long_device.restype = C.c_int
    lib.psa_align_long_device.argtypes = [vp, vp, vp, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_uint,
                                          vp, vp, C.c_size_t, vp]
    lib.psa_align_pair_banded.restype = C.c_int
    lib.psa_align_pair_banded.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int,
                                          C.c_uint, C.POINTER(_Result)]
    lib.psa_align_long_banded_device.restype = C.c_int
    lib.psa_align_long_banded_device.argtypes = [vp, vp, vp, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint,
                                                 vp, vp, C.c_size_t, vp]
    lib.psa_align_batch_guided.restype = C.c_int
    lib.psa_align_batch_guided.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_size_t, C.c_size_t, vp, vp, vp, C.c_size_t,
                                           C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint, vp, vp, C.c_size_t]
    lib.psa_align_batch_guided_device.restype = C.c_int
    lib.psa_align_batch_guided_device.argtypes = [vp, vp, vp, vp, vp, vp, vp, C.c_size_t, C.c_int, C.c_int, vp, vp, vp, C.c_int,
                                                  C.c_int, C.c_int, C.c_int, C.c_uint, vp, vp, C.c_size_t, vp]
    lib.psa_align_pair_guided.restype = C.c_int
    lib.psa_align_pair_guided.argtypes = [vp, C.c_char_p, C.c_char_p, C.c_size_t, C.c_size_t, vp, C.c_size_t, C.c_int, C.c_int,
                                          C.c_int, C.c_int, C.c_uint, C.POINTER(_Result)]
    lib.psa_xbuf_bytes.restype = C.c_size_t
    lib.psa_xbuf_bytes.argtypes = [C.c_size_t]
    lib.psa_xbuf_create.restype = C.c_int
    lib.psa_xbuf_create.argtypes = [vp, C.c_size_t, C.POINTER(vp), C.c_char_p]
    lib.psa_xbuf_open.restype = C.c_int
    lib.psa_xbuf_open.argtypes = [vp, C.c_char_p, C.POINTER(vp)]
    lib.psa_xbuf_close.restype = C.c_int
    lib.psa_xbuf_close.argtypes = [vp, vp]
    lib.psa_xbuf_destroy.restype = C.c_int
    lib.psa_xbuf_destroy.argtypes = [vp, vp]
    lib.psa_long_panel_strips.restype = C.c_int
    lib.psa_long_panel_strips.argtypes = [vp]
    lib.psa_long_strip_columns.restype = C.c_int
    lib.psa_long_strip_columns.argtypes = [vp]
    lib.psa_align_long_cyclic_device.restype = C.c_int
    lib.psa_align_long_cyclic_device.argtypes = [vp, vp, vp, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                                 C.c_int, C.c_size_t, vp, vp, vp, vp]
    lib.psa_ops_unpack.restype = None
    lib.psa_ops_unpack.argtypes = [vp, i32, vp]
    lib.psa_render_rows.restype = None
    lib.psa_render_rows.argtypes = [C.c_char_p, C.c_char_p, vp, i64, i64, i64, vp, vp]
    lib.psa_peak_int_ops.restype = C.c_int
    lib.psa_peak_int_ops.argtypes = [vp, C.c_int, C.POINTER(C.c_double), C.POINTER(C.c_double)]
    _lib = lib
    return lib


EXPORTS = ["psa_ctx_create", "psa_ctx_destroy", "psa_last_error", "psa_launch_count", "psa_align_pair", "psa_align_pair_typed", "psa_align_partition", "psa_align_long_partitioned", "psa_similarity_batch", "psa_similarity_batch_device",
           "psa_result_free", "psa_align_batch", "psa_align_batch_device", "psa_align_batch_banded", "psa_align_batch_banded_device", "psa_pack_bases", "psa_pack_reads", "psa_align_batch_packed", "psa_align_long_device", "psa_align_pair_banded", "psa_align_long_banded_device",
           "psa_align_batch_guided", "psa_align_batch_guided_device", "psa_align_pair_guided", "psa_xbuf_bytes", "psa_xbuf_create", "psa_xbuf_open", "psa_xbuf_close",
           "psa_xbuf_destroy", "psa_long_panel_strips", "psa_long_strip_columns", "psa_align_long_cyclic_device", "psa_ops_unpack", "psa_render_rows",
           "psa_peak_int_ops"]


def pack_pairs(seqs: Sequence[bytes]):
    """Concatenate sequences back to back -> (uint8 bases, int64 offsets, int32 lengths)."""
    lens = np.fromiter((len(s) for s in seqs), dtype=np.int32, count=len(seqs))
    offs = np.zeros(len(seqs), dtype=np.int64)
    if len(seqs) > 1:
        np.cumsum(lens[:-1], out=offs[1:])
    bases = np.frombuffer(b"".join(seqs), dtype=np.uint8).copy() if len(seqs) else np.zeros(0, np.uint8)
    return bases, offs, lens


def pack_bases(seq: bytes):
    """psa_pack_bases: ACGT bytes -> (2-bit words, number of bytes that are not ACGT)."""
    lib = load_library()
    out = np.zeros((len(seq) + 15) // 16, dtype=np.uint32)
    buf = np.frombuffer(seq, dtype=np.uint8)
    bad = lib.psa_pack_bases(buf.ctypes.data if len(seq) else None, len(seq), out.ctypes.data if len(out) else None)
    return out, int(bad)


def pack_reads(reads: np.ndarray, threads: int = 0, out: Optional[np.ndarray] = None):
    """psa_pack_reads: a [n, L] uint8 matrix of ASCII reads (rows may be strided) -> ([n, ceil(L/16)] uint32 in the
    layout psa_align_batch_packed takes, number of bytes that are not ACGT).  Multi-threaded host code, no GPU."""
    lib = load_library()
    n, L = reads.shape
    assert reads.dtype == np.uint8 and (L == 0 or reads.strides[1] == 1)
    W = (L + 15) // 16
    if out is None:
        out = np.zeros((n, W), dtype=np.uint32)
    assert out.shape == (n, W) and out.dtype == np.uint32 and out.flags.c_contiguous
    if n == 0 or L == 0:
        return out, 0
    bad = lib.psa_pack_reads(reads.ctypes.data, n, L, reads.strides[0], out.ctypes.data, threads)
    return out, int(bad)


def pack_reads_2bit(reads: np.ndarray) -> np.ndarray:
    """Vectorised form of psa_pack_bases for a [n, L] uint8 matrix of ACGT letters -> [n, ceil(L/16)] uint32
    (the fixed-stride layout psa_align_batch_packed takes)."""
    n, L = reads.shape
    W = (L + 15) // 16
    codes = np.zeros((n, W * 16), dtype=np.uint32)
    codes[:, :L] = (reads >> 1) & 3
    codes = codes.reshape(n, W, 16)
    return np.ascontiguousarray((codes << (2 * np.arange(16, dtype=np.uint32))[None, None, :]).sum(axis=2, dtype=np.uint32))


def compact_ops_offsets(items: np.ndarray) -> np.ndarray:
    """Word offset of every pair's ops in a PSA_OPS_COMPACT buffer: the running sum of ceil(aln_len/16)."""
    words = (items["aln_len"].astype(np.int64) + 15) >> 4
    out = np.zeros(len(items) + 1, dtype=np.int64)
    np.cumsum(words, out=out[1:])
    return out


def pack_anchors(anchors: Sequence) -> tuple:
    """Per-pair anchor chains ((K_k, 2) arrays of (i, j), or lists of pairs) -> (psa_anchor array [total, 2] int32,
    int64 offsets, int32 counts), the layout psa_align_batch_guided takes."""
    chains = [np.asarray(c, dtype=np.int64).reshape(-1, 2) for c in anchors]
    cnt = np.array([len(c) for c in chains], dtype=np.int32)
    off = np.zeros(len(chains), dtype=np.int64)
    if len(chains) > 1:
        np.cumsum(cnt[:-1], out=off[1:])
    flat = np.concatenate(chains) if chains and cnt.sum() else np.zeros((0, 2), np.int64)
    if flat.size and (flat.min() < -2 ** 31 or flat.max() >= 2 ** 31):
        raise ValueError("anchor coordinates must fit int32")
    return np.ascontiguousarray(flat, dtype=np.int32), off, cnt


def unpack_ops(words: np.ndarray, aln_len: int) -> bytes:
    """2-bit traceback-order words -> forward-order state bytes (1/2/3)."""
    if aln_len == 0:
        return b""
    w = np.ascontiguousarray(words, dtype=np.uint32)
    k = np.arange(aln_len)
    codes = (w[k >> 4] >> (2 * (k & 15)).astype(np.uint32)) & 3
    return codes[::-1].astype(np.uint8).tobytes()


def render_rows(a: bytes, b: bytes, ops: bytes, start_i: int, start_j: int):
    lib = load_library()
    n = len(ops)
    ra, rb = C.create_string_buffer(n + 1), C.create_string_buffer(n + 1)
    buf = (C.c_uint8 * max(n, 1)).from_buffer_copy(ops if n else b"\0")
    lib.psa_render_rows(a, b, C.addressof(buf), n, start_i, start_j, C.addressof(ra), C.addressof(rb))
    return ra.raw[:n], rb.raw[:n]


class PairResult:
    __slots__ = ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j", "start_i", "start_j", "ops", "row_a",
                 "row_b")

    def __repr__(self):
        return f"PairResult(score={self.score}, corner=({self.t1},{self.t2},{self.t3}), len={len(self.ops)})"


class Context:
    """psa_ctx: one per (host thread, device)."""

    def __init__(self, device: int = 0):
        self._lib = load_library()
        self._h = C.c_void_p()
        rc = self._lib.psa_ctx_create(device, C.byref(self._h))
        if rc != 0:
            raise PsaError(rc, self._lib.psa_last_error(None).decode())
        self.device = device

    def close(self):
        if self._h:
            self._lib.psa_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise PsaError(rc, self._lib.psa_last_error(self._h).decode())

    def set_option(self, name: str, value: int):
        """Test / measurement hook (csrc/psa_internal.h): kernel-variant selection and timing switches."""
        self._check(self._lib.psa_ctx_set_option(self._h, name.encode(), int(value)))

    @property
    def launches(self) -> int:
        return int(self._lib.psa_launch_count(self._h))

    def align_pair(self, a: bytes, b: bytes, mode: int = GLOBAL, g: int = 1, h: int = 2,
                   traceback: bool = True, start_type: int = -1, end_type: int = -1) -> PairResult:
        res = _Result()
        flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        if start_type != -1 or end_type != -1:
            self._check(self._lib.psa_align_pair_typed(self._h, a, b, len(a), len(b), start_type, end_type, g, h, flags,
                                                       C.byref(res)))
        else:
            self._check(self._lib.psa_align_pair(self._h, a, b, len(a), len(b), mode, g, h, flags, C.byref(res)))
        return self._take(res, traceback)

    def _take(self, res, traceback: bool = True) -> PairResult:
        out = PairResult()
        for f in ("t1", "t2", "t3", "score", "end_state", "end_i", "end_j", "start_i", "start_j"):
            setattr(out, f, getattr(res, f))
        n = res.aln_len
        out.ops = bytes(res.ops[:n]) if traceback and n else b""
        out.row_a = C.string_at(res.row_a, n) if traceback and res.row_a else b""
        out.row_b = C.string_at(res.row_b, n) if traceback and res.row_b else b""
        self._lib.psa_result_free(C.byref(res))
        return out

    def similarity_batch(self, bases_a: np.ndarray, off_a: np.ndarray, len_a: np.ndarray, bases_b: np.ndarray,
                         off_b: np.ndarray, len_b: np.ndarray) -> np.ndarray:
        """sequence_similarity of every pair (psa_similarity_batch, host buffers)."""
        bases_a = np.ascontiguousarray(bases_a, dtype=np.uint8)
        bases_b = np.ascontiguousarray(bases_b, dtype=np.uint8)
        off_a = np.ascontiguousarray(off_a, dtype=np.int64)
        off_b = np.ascontiguousarray(off_b, dtype=np.int64)
        len_a = np.ascontiguousarray(len_a, dtype=np.int32)
        len_b = np.ascontiguousarray(len_b, dtype=np.int32)
        out = np.zeros(len(len_a), dtype=np.float64)
        self._check(self._lib.psa_similarity_batch(self._h, bases_a.ctypes.data, off_a.ctypes.data, len_a.ctypes.data,
                                                   bases_b.ctypes.data, off_b.ctypes.data, len_b.ctypes.data, len(len_a),
                                                   bases_a.size, bases_b.size, out.ctypes.data))
        return out

    def similarity_batch_device(self, d_bases_a: int, d_off_a: int, d_len_a: int, d_bases_b: int, d_off_b: int,
                                d_len_b: int, n_pairs: int, max_len: int, d_out: int, stream: int = 0):
        self._check(self._lib.psa_similarity_batch_device(self._h, d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b,
                                                          n_pairs, max_len, d_out, stream or None))

    def align_partition(self, a: bytes, b: bytes, points, g: int = 1, h: int = 2) -> PairResult:
        """optimal_alignment over a partition (psa_align_partition): points = [(i, j, t), ...]."""
        bp = np.zeros(len(points), dtype=BP_DTYPE)
        for k, (i, j, t) in enumerate(points):
            bp[k] = (i, j, t, 0)
        res = _Result()
        self._check(self._lib.psa_align_partition(self._h, a, b, len(a), len(b), bp.ctypes.data, len(points), g, h,
                                                  C.byref(res)))
        return self._take(res)

    def align_long_partitioned(self, a: bytes, b: bytes, pieces: int, g: int = 1, h: int = 2):
        """psa_align_long_partitioned: partition finder + stitched complete alignment.  Returns (PairResult, crossings)."""
        res = _Result()
        bp = np.zeros(max(pieces, 1), dtype=BP_DTYPE)
        nbp = C.c_size_t(0)
        self._check(self._lib.psa_align_long_partitioned(self._h, a, b, len(a), len(b), g, h, pieces, C.byref(res), bp.ctypes.data,
                                                         len(bp), C.byref(nbp)))
        return self._take(res), [(int(x["i"]), int(x["j"]), int(x["t"])) for x in bp[:nbp.value]]

    def align_batch(self, bases_a: np.ndarray, off_a: np.ndarray, len_a: np.ndarray, bases_b: np.ndarray,
                    off_b: np.ndarray, len_b: np.ndarray, mode: int = GLOBAL, g: int = 1, h: int = 2,
                    traceback: bool = True, items: Optional[np.ndarray] = None, ops: Optional[np.ndarray] = None):
        """Host-buffer batch call (psa_align_batch).  Returns (items structured array, ops words
        [n_pairs, stride] or None)."""
        n = len(len_a)
        bases_a = np.ascontiguousarray(bases_a, dtype=np.uint8)
        bases_b = np.ascontiguousarray(bases_b, dtype=np.uint8)
        off_a = np.ascontiguousarray(off_a, dtype=np.int64)
        off_b = np.ascontiguousarray(off_b, dtype=np.int64)
        len_a = np.ascontiguousarray(len_a, dtype=np.int32)
        len_b = np.ascontiguousarray(len_b, dtype=np.int32)
        if items is None:
            items = np.zeros(n, dtype=ITEM_DTYPE)
        stride = 0
        if traceback:
            stride = (int(len_a.max(initial=0)) + int(len_b.max(initial=0)) + 15) // 16 + 1
            if ops is None:
                ops = np.zeros((n, stride), dtype=np.uint32)
            else:
                stride = ops.shape[1]
        flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_batch(
            self._h, bases_a.ctypes.data, off_a.ctypes.data, len_a.ctypes.data, bases_b.ctypes.data,
            off_b.ctypes.data, len_b.ctypes.data, n, bases_a.size, bases_b.size, mode, g, h, flags,
            items.ctypes.data, ops.ctypes.data if traceback else None, stride))
        return items, (ops if traceback else None)

    def align_batch_packed(self, a2: np.ndarray, b2: np.ndarray, len_a: int, len_b: int, mode: int = LOCAL, g: int = 1, h: int = 2,
                           traceback: bool = True, items: Optional[np.ndarray] = None, ops: Optional[np.ndarray] = None,
                           compact: bool = False):
        """psa_align_batch_packed: fixed-stride 2-bit reads ([n, ceil(len/16)] uint32 each) -> (16-byte records, op words).
        compact=True (PSA_OPS_COMPACT): the op words come back to back in pair order in ops.reshape(-1); pair k starts at
        compact_ops_offsets(items)[k]."""
        n = a2.shape[0]
        assert a2.dtype == np.uint32 and b2.dtype == np.uint32 and a2.flags.c_contiguous and b2.flags.c_contiguous
        if items is None:
            items = np.zeros(n, dtype=PACKED_ITEM_DTYPE)
        stride = 0
        if traceback:
            stride = (len_a + len_b + 15) // 16 + 1 if ops is None else ops.shape[1]
            if ops is None:
                ops = np.zeros((n, stride), dtype=np.uint32)
        flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0) | (OPS_COMPACT if compact and traceback else 0)
        self._check(self._lib.psa_align_batch_packed(self._h, a2.ctypes.data, b2.ctypes.data, n, len_a, len_b, mode, g, h, flags,
                                                     items.ctypes.data, ops.ctypes.data if traceback else None, stride))
        return items, (ops if traceback else None)

    def align_batch_device(self, d_bases_a: int, d_off_a: int, d_len_a: int, d_bases_b: int, d_off_b: int,
                           d_len_b: int, n_pairs: int, max_len_a: int, max_len_b: int, d_items: int,
                           d_ops: int = 0, ops_stride_words: int = 0, mode: int = GLOBAL, g: int = 1, h: int = 2,
                           traceback: bool = True, stream: int = 0):
        """Device-resident batch call: all arguments are raw device pointers / a raw cudaStream_t."""
        flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_batch_device(
            self._h, d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b, n_pairs, max_len_a, max_len_b,
            mode, g, h, flags, d_items, d_ops or None, ops_stride_words, stream or None))

    def align_batch_banded(self, bases_a: np.ndarray, off_a: np.ndarray, len_a: np.ndarray, bases_b: np.ndarray,
                           off_b: np.ndarray, len_b: np.ndarray, band: int, mode: int = GLOBAL, g: int = 1, h: int = 2,
                           traceback: bool = True, ops: Optional[np.ndarray] = None, flags: Optional[int] = None):
        """psa_align_batch_banded: align_batch inside the diagonal band of half-width `band`.  Returns (items, ops words
        [n_pairs, stride] or None)."""
        n = len(len_a)
        bases_a = np.ascontiguousarray(bases_a, dtype=np.uint8)
        bases_b = np.ascontiguousarray(bases_b, dtype=np.uint8)
        off_a = np.ascontiguousarray(off_a, dtype=np.int64)
        off_b = np.ascontiguousarray(off_b, dtype=np.int64)
        len_a = np.ascontiguousarray(len_a, dtype=np.int32)
        len_b = np.ascontiguousarray(len_b, dtype=np.int32)
        items = np.zeros(n, dtype=ITEM_DTYPE)
        stride = 0
        if traceback:
            if ops is None:
                stride = (int(len_a.max(initial=0)) + int(len_b.max(initial=0)) + 15) // 16 + 1
                ops = np.zeros((n, stride), dtype=np.uint32)
            stride = ops.shape[1]
        if flags is None:
            flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_batch_banded(
            self._h, bases_a.ctypes.data, off_a.ctypes.data, len_a.ctypes.data, bases_b.ctypes.data,
            off_b.ctypes.data, len_b.ctypes.data, n, bases_a.size, bases_b.size, mode, g, h, band, flags,
            items.ctypes.data, ops.ctypes.data if traceback else None, stride))
        return items, (ops if traceback else None)

    def align_batch_banded_device(self, d_bases_a: int, d_off_a: int, d_len_a: int, d_bases_b: int, d_off_b: int,
                                  d_len_b: int, n_pairs: int, max_len_a: int, max_len_b: int, band: int, d_items: int,
                                  d_ops: int = 0, ops_stride_words: int = 0, mode: int = GLOBAL, g: int = 1, h: int = 2,
                                  traceback: bool = True, stream: int = 0, flags: Optional[int] = None):
        """Device-resident banded batch call (psa_align_batch_banded_device): raw device pointers / cudaStream_t."""
        if flags is None:
            flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_batch_banded_device(
            self._h, d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b, n_pairs, max_len_a, max_len_b,
            mode, g, h, band, flags, d_items, d_ops or None, ops_stride_words, stream or None))

    def align_batch_guided(self, bases_a: np.ndarray, off_a: np.ndarray, len_a: np.ndarray, bases_b: np.ndarray,
                           off_b: np.ndarray, len_b: np.ndarray, anchors: Sequence, band: int, mode: int = GLOBAL, g: int = 1,
                           h: int = 2, traceback: bool = True, ops: Optional[np.ndarray] = None, flags: Optional[int] = None):
        """psa_align_batch_guided: align_batch_banded with each pair's band around its anchor chain; anchors[k] is pair k's
        chain, a (K_k, 2) array of (i, j).  Returns (items, ops words [n_pairs, stride] or None)."""
        n = len(len_a)
        bases_a = np.ascontiguousarray(bases_a, dtype=np.uint8)
        bases_b = np.ascontiguousarray(bases_b, dtype=np.uint8)
        off_a = np.ascontiguousarray(off_a, dtype=np.int64)
        off_b = np.ascontiguousarray(off_b, dtype=np.int64)
        len_a = np.ascontiguousarray(len_a, dtype=np.int32)
        len_b = np.ascontiguousarray(len_b, dtype=np.int32)
        anc, off_anc, n_anc = pack_anchors(anchors)
        if len(n_anc) != n:
            raise ValueError("one anchor chain per pair")
        items = np.zeros(n, dtype=ITEM_DTYPE)
        stride = 0
        if traceback:
            if ops is None:
                stride = (int(len_a.max(initial=0)) + int(len_b.max(initial=0)) + 15) // 16 + 1
                ops = np.zeros((n, stride), dtype=np.uint32)
            stride = ops.shape[1]
        if flags is None:
            flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_batch_guided(
            self._h, bases_a.ctypes.data, off_a.ctypes.data, len_a.ctypes.data, bases_b.ctypes.data,
            off_b.ctypes.data, len_b.ctypes.data, n, bases_a.size, bases_b.size, anc.ctypes.data if len(anc) else None,
            off_anc.ctypes.data, n_anc.ctypes.data, len(anc), mode, g, h, band, flags,
            items.ctypes.data, ops.ctypes.data if traceback else None, stride))
        return items, (ops if traceback else None)

    def align_batch_guided_device(self, d_bases_a: int, d_off_a: int, d_len_a: int, d_bases_b: int, d_off_b: int,
                                  d_len_b: int, n_pairs: int, max_len_a: int, max_len_b: int, d_anchors: int, d_off_anc: int,
                                  d_n_anc: int, band: int, d_items: int, d_ops: int = 0, ops_stride_words: int = 0,
                                  mode: int = GLOBAL, g: int = 1, h: int = 2, traceback: bool = True, stream: int = 0,
                                  flags: Optional[int] = None):
        """psa_align_batch_guided_device: raw device pointers / cudaStream_t; anchors as pack_anchors lays them out.  A pair
        whose chain is invalid gets the rejected record (end_state 0)."""
        if flags is None:
            flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_batch_guided_device(
            self._h, d_bases_a, d_off_a, d_len_a, d_bases_b, d_off_b, d_len_b, n_pairs, max_len_a, max_len_b,
            d_anchors or None, d_off_anc or None, d_n_anc or None, mode, g, h, band, flags, d_items, d_ops or None,
            ops_stride_words, stream or None))

    def align_pair_guided(self, a: bytes, b: bytes, anchors, band: int, mode: int = GLOBAL, g: int = 1, h: int = 2,
                          traceback: bool = True, flags: Optional[int] = None) -> PairResult:
        """psa_align_pair_guided: one pair inside the band around its anchor chain ((K, 2) array of (i, j)), over the whole
        GPU."""
        anc, _, cnt = pack_anchors([anchors])
        res = _Result()
        if flags is None:
            flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_pair_guided(self._h, a, b, len(a), len(b), anc.ctypes.data if len(anc) else None,
                                                    int(cnt[0]), mode, g, h, band, flags, C.byref(res)))
        return self._take(res, traceback)

    def align_long_device(self, d_a: int, d_b: int, m: int, n: int, d_item: int, d_ops: int = 0, ops_words: int = 0,
                          mode: int = GLOBAL, g: int = 1, h: int = 2, traceback: bool = False, stream: int = 0):
        """One long pair resident in device memory (raw pointers); asynchronous on `stream`."""
        flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_long_device(self._h, d_a, d_b, m, n, mode, g, h, flags, d_item, d_ops or None,
                                                    ops_words, stream or None))

    def align_pair_banded(self, a: bytes, b: bytes, band: int, mode: int = GLOBAL, g: int = 1, h: int = 2,
                          traceback: bool = True, flags: Optional[int] = None) -> PairResult:
        """psa_align_pair_banded: one pair inside the diagonal band of half-width `band`, over the whole GPU."""
        res = _Result()
        if flags is None:
            flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_pair_banded(self._h, a, b, len(a), len(b), mode, g, h, band, flags, C.byref(res)))
        return self._take(res, traceback)

    def align_long_banded_device(self, d_a: int, d_b: int, m: int, n: int, band: int, d_item: int, d_ops: int = 0,
                                 ops_words: int = 0, mode: int = GLOBAL, g: int = 1, h: int = 2, traceback: bool = False,
                                 stream: int = 0, flags: Optional[int] = None):
        """psa_align_long_banded_device: one banded pair resident in device memory (raw pointers); asynchronous on `stream`."""
        if flags is None:
            flags = WANT_SCORE | (WANT_TRACEBACK if traceback else 0)
        self._check(self._lib.psa_align_long_banded_device(self._h, d_a, d_b, m, n, mode, g, h, band, flags, d_item,
                                                           d_ops or None, ops_words, stream or None))

    # ---- one long pair over several GPUs: block-cyclic systolic panels (config 4) ----
    def xbuf_create(self, m_cap: int):
        """Allocates this rank's incoming inter-GPU boundary buffer; returns (device pointer, 64-byte IPC handle)."""
        ptr = C.c_void_p()
        handle = C.create_string_buffer(64)
        self._check(self._lib.psa_xbuf_create(self._h, m_cap, C.byref(ptr), handle))
        return ptr.value, handle.raw

    def xbuf_open(self, handle: bytes) -> int:
        ptr = C.c_void_p()
        self._check(self._lib.psa_xbuf_open(self._h, handle, C.byref(ptr)))
        return ptr.value

    def xbuf_close(self, ptr: int):
        self._check(self._lib.psa_xbuf_close(self._h, ptr))

    def xbuf_destroy(self, ptr: int):
        self._check(self._lib.psa_xbuf_destroy(self._h, ptr))

    @property
    def long_panel_strips(self) -> int:
        return int(self._lib.psa_long_panel_strips(self._h))

    @property
    def long_strip_columns(self) -> int:
        return int(self._lib.psa_long_strip_columns(self._h))

    def align_long_cyclic_device(self, d_a: int, d_b: int, m: int, n: int, rank: int, world: int, panel_strips: int,
                                 d_item: int, m_cap: int = 0, d_xin: int = 0, d_xout_peer: int = 0, mode: int = LOCAL, g: int = 1,
                                 h: int = 2, stream: int = 0):
        self._check(self._lib.psa_align_long_cyclic_device(self._h, d_a, d_b, m, n, rank, world, panel_strips, mode, g, h,
                                                           m_cap or m, d_xin or None, d_xout_peer or None, d_item, stream or None))

    def peak_int_ops(self, kind: int):
        v, ms = C.c_double(), C.c_double()
        self._check(self._lib.psa_peak_int_ops(self._h, kind, C.byref(v), C.byref(ms)))
        return v.value, ms.value
