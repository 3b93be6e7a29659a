"""The chunked host pipeline of psa_align_batch (byte input, batches larger than one chunk) and the chunked
device-resident entry: the same results as the un-chunked and the generic routes, with the launch counts the chunk
schedule implies."""
import functools

import numpy as np
import pytest
import torch

import cse305_parallel_sequence_alignment_b200 as psa
from cse305_parallel_sequence_alignment_b200.capi import ITEM_DTYPE
from oracle import pyoracle as po

pytestmark = pytest.mark.gpu

ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)
PROTEIN = b"ARNDCQEGHILKMFPSTWYV"


def _chunk_sizes(chunk, n):
    """The host pipeline's chunk schedule: full chunks in the middle, ramped down to chunk/8 at both ends when the
    batch is long enough and the chunks are at least 8192 pairs."""
    ramp = [chunk // 8, chunk // 4, chunk // 2]
    if n >= 2 * sum(ramp) + chunk and chunk >= 8192:
        mid = n - 2 * sum(ramp)
        return ramp + [min(chunk, mid - p) for p in range(0, mid, chunk)] + ramp[::-1]
    return [min(chunk, n - p) for p in range(0, n, chunk)]


def _walk_launches(tb, ckpt):
    """Launches of one chunk's traceback: the code walk, or the two perm passes + the tile-recompute walk."""
    return 0 if not tb else (3 if ckpt else 1)


@functools.lru_cache(maxsize=None)
def _batch(n, max_m, max_n, seed):
    """n ragged pairs laid out back to back (A up to max_m, B up to max_n; pair 0 has both maxima): similar pairs,
    shifted pairs and random pairs, and members the packed fill must flag -- N, lower case, empty, another
    alphabet -- spread over the chunks."""
    rng = np.random.default_rng(seed)
    la, lb = rng.integers(1, max_m + 1, size=n), rng.integers(1, max_n + 1, size=n)
    la[0], lb[0] = max_m, max_n
    A = ACGT[rng.integers(0, 4, size=(n, max_m))]
    B = ACGT[rng.integers(0, 4, size=(n, max_n))]
    k = min(max_m, max_n)
    B[0::4, :k] = A[0::4, :k]
    B[2::4, :k - 3] = A[2::4, 3:k]
    mut = rng.random(B.shape) < 0.06
    B[mut] = ACGT[rng.integers(0, 4, size=int(mut.sum()))]
    As = [A[q, :la[q]].tobytes() for q in range(n)]
    Bs = [B[q, :lb[q]].tobytes() for q in range(n)]
    flagged = list(range(5, n, 997))
    for j, q in enumerate(flagged):
        kind = j % 4
        if kind == 0:
            As[q] = As[q][: len(As[q]) // 2] + b"N" + As[q][len(As[q]) // 2 + 1:]
        elif kind == 1:
            Bs[q] = Bs[q].lower()
        elif kind == 2:
            (As if j % 8 == 2 else Bs)[q] = b""
        else:
            As[q] = bytes(PROTEIN[int(x)] for x in rng.integers(0, len(PROTEIN), size=len(As[q])))
    return As, Bs, flagged


def _assert_same(items, ops, ref_items, ref_ops, tb, what):
    for f in ITEM_DTYPE.names:
        assert np.array_equal(items[f], ref_items[f]), (what, f, np.flatnonzero(items[f] != ref_items[f])[:8])
    if tb:
        words = (items["aln_len"] + 15) // 16         # the words that carry ops (the tail of a stride is unspecified)
        mask = np.arange(ops.shape[1])[None, :] < words[:, None]
        assert np.array_equal(ops[mask], ref_ops[mask]), what


def _oracle_sample(As, Bs, flagged, items, ops, mode, tb):
    for q in list(range(0, len(As), 331)) + flagged:
        if not As[q] or not Bs[q]:
            continue
        w = po.align(As[q], Bs[q], 1, 2, mode=mode)
        it = items[q]
        assert (it["score"], it["end_i"], it["end_j"]) == (w.score, w.end_i, w.end_j), q
        if mode == psa.GLOBAL:
            assert (it["t1"], it["t2"], it["t3"], it["end_state"]) == (w.t1, w.t2, w.t3, w.end_state), q
        if tb:
            assert (it["start_i"], it["start_j"]) == (w.start_i, w.start_j), q
            assert psa.unpack_ops(ops[q], int(it["aln_len"])) == w.ops, q


# (pack_chunk, pairs): several 1 024-pair chunks and a short last one; ramped 8 192-pair chunks (1 024, 2 048, 4 096,
# 8 192, 1 000, 4 096, 2 048, 1 024)
CHUNKINGS = [(1024, 5000), (8192, 23528)]
# (traceback, pack_traceback, pack_serial_fills)
VARIANTS = [(False, 0, 0), (False, 0, 1), (True, 0, 0), (True, 0, 1), (True, 1, 0), (True, 1, 1)]


@pytest.mark.parametrize("chunking", CHUNKINGS, ids=["chunk1024", "chunk8192_ramp"])
@pytest.mark.parametrize("shape", [(150, 150), (300, 250)])
@pytest.mark.parametrize("mode", [psa.LOCAL, psa.GLOBAL])
def test_byte_pipeline_equals_unchunked_and_generic(mode, shape, chunking):
    """psa_align_batch through the chunked host pipeline (both traceback flavours, fills serialised or not, flagged
    members in several chunks) == the same batch with pipeline = 0 (all copies first, the device entry) == the
    generic int32 kernel (pack = 0); a sample == the oracle."""
    chunk, n = chunking
    As, Bs, flagged = _batch(n, shape[0], shape[1], 1000 + shape[1])
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    sizes = _chunk_sizes(chunk, n)
    assert sum(sizes) == n and len(sizes) > 4
    c = psa.Context(0)
    try:
        c.set_option("pack_chunk", chunk)
        ref = {}
        c.set_option("pack", 0)
        for tb in (False, True):
            l0 = c.launches
            ref[tb] = c.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=tb)
            assert c.launches - l0 == 1
        c.set_option("pack", 1)
        for tb, ckpt, serial in VARIANTS:
            what = dict(tb=tb, ckpt=ckpt, serial=serial)
            c.set_option("pack_traceback", ckpt)
            c.set_option("pack_serial_fills", serial)
            per_chunk = 2 + _walk_launches(tb, ckpt)        # fill + walk + the generic kernel on the flagged members
            l0 = c.launches
            items, ops = c.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=tb)
            assert c.launches - l0 == len(sizes) * per_chunk, what
            _assert_same(items, ops, *ref[tb], tb, what)
            c.set_option("pipeline", 0)
            l0 = c.launches
            items_u, ops_u = c.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=tb)
            assert c.launches - l0 == (-(-n // chunk) if tb else 1) * per_chunk, what
            c.set_option("pipeline", 1)
            _assert_same(items_u, ops_u, items, ops, tb, what)
            if not ckpt and not serial:
                _oracle_sample(As, Bs, flagged, items, ops, mode, tb)
    finally:
        c.close()


@pytest.mark.parametrize("ckpt", [0, 1])
@pytest.mark.parametrize("mode", [psa.LOCAL, psa.GLOBAL])
def test_device_entry_chunks_on_side_stream(mode, ckpt):
    """psa_align_batch_device over several 1 024-pair chunks on a torch side stream: == the host entry, and ready
    once that stream alone is synchronised (the library's own streams join it)."""
    n, chunk = 5000, 1024
    As, Bs, _ = _batch(n, 150, 150, 1150)
    ba, oa, la = psa.pack_pairs(As)
    bb, ob, lb = psa.pack_pairs(Bs)
    c = psa.Context(0)
    try:
        c.set_option("pack_chunk", chunk)
        c.set_option("pack_traceback", ckpt)
        want_items, want_ops = c.align_batch(ba, oa, la, bb, ob, lb, mode, 1, 2, traceback=True)
        stride = want_ops.shape[1]
        d = [torch.from_numpy(x).cuda() for x in (ba, oa, la, bb, ob, lb)]
        d_items = torch.zeros(n * ITEM_DTYPE.itemsize // 4, dtype=torch.int32, device="cuda")
        d_ops = torch.zeros(n * stride, dtype=torch.int32, device="cuda")
        torch.cuda.synchronize()
        stream = torch.cuda.Stream()
        l0 = c.launches
        c.align_batch_device(*(x.data_ptr() for x in d), n, int(la.max()), int(lb.max()), d_items.data_ptr(),
                             d_ops.data_ptr(), stride, mode, 1, 2, True, stream.cuda_stream)
        assert c.launches - l0 == -(-n // chunk) * (2 + _walk_launches(True, ckpt))
        stream.synchronize()
        items = d_items.cpu().numpy().view(ITEM_DTYPE)
        ops = d_ops.cpu().numpy().view(np.uint32).reshape(n, stride)
        _assert_same(items, ops, want_items, want_ops, True, "device entry")
    finally:
        c.close()
