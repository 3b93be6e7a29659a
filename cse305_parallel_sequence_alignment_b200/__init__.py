"""B200-native pairwise-alignment hot path (Gotoh fill + traceback) behind a C-ABI.

The product is libpsa.so (hand-written sm_100a CUDA, include/psa.h).  This package is the thin
Python doorway used by the tests, bench.py and __graft_entry__: it loads the shared library with
ctypes and fails loudly if the library or a CUDA device is missing -- there is no CPU fallback.
"""
from .capi import (GLOBAL, LOCAL, WANT_SCORE, WANT_TRACEBACK, OPS_COMPACT, compact_ops_offsets, BatchItem, Context, PsaError, build_library,
                   library_path, load_library, pack_anchors, pack_pairs, unpack_ops, render_rows, pack_bases, pack_reads, pack_reads_2bit)

__all__ = ["GLOBAL", "LOCAL", "WANT_SCORE", "WANT_TRACEBACK", "OPS_COMPACT", "compact_ops_offsets", "BatchItem", "Context", "PsaError",
           "build_library", "library_path", "load_library", "pack_anchors", "pack_pairs", "unpack_ops", "render_rows", "pack_bases", "pack_reads", "pack_reads_2bit"]
