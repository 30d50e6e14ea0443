"""Beam-search reorder without a GPU: the kvc_batch_region records the slab and its followers pack, the index checks,
and the C ABI's refusals (all before any CUDA call)."""

import ctypes

import pytest
import torch

from kvcompress import H2OScoreSlab, KVSlabCache, SnapKVQueryWindow, _engine

INVALID, UNSUPPORTED = 1, 2


def host_slab(L=3, B=4, H=2, D=8, cap=16, dtype=torch.float16, pinned=False):
    """A KVSlabCache over host tensors laid out as the constructor lays them out (pitch = capacity + 8 here)."""
    slab = KVSlabCache.__new__(KVSlabCache)
    slab.num_layers, slab.batch, slab.heads, slab.head_dim, slab.capacity = L, B, H, D, cap
    slab.dtype, slab.device, slab.pinned = dtype, torch.device("cuda", 0), pinned
    slab.k = torch.zeros((L, B, H, cap + 8, D), dtype=dtype)[:, :, :, :cap]
    slab.v = torch.zeros((L, B, H, cap + 8, D), dtype=dtype)[:, :, :, :cap]
    slab.n = torch.zeros((L, B, H, cap), dtype=dtype)
    slab.lengths = [0] * L
    slab._reorder_recs = None
    return slab


def unpack(recs):
    return [_engine._REGION.unpack_from(recs, i) for i in range(0, len(recs), _engine._REGION.size)]


def test_slab_records_follow_the_lengths():
    slab = host_slab()
    slab.lengths = [5, 0, 16]
    e, D, pitch = 2, 8, 24
    regions = unpack(slab._reorder_records())
    assert len(regions) == 9                                   # K, V, norms of every layer
    k0, v0, n0, k1, v1, n1, k2, _, n2 = regions
    assert k0 == (slab.k[0].data_ptr(), 2 * pitch * D * e, pitch * D * e, 5 * D * e, 2, e)
    assert v0[0] == slab.v[0].data_ptr() and v0[3] == 5 * D * e
    assert n0 == (slab.n[0].data_ptr(), 2 * 16 * e, 16 * e, 5 * e, 2, e)
    assert k1[3] == v1[3] == n1[3] == 0                        # the empty layer moves nothing
    assert k2[3] == 16 * D * e and n2[3] == 16 * e
    # a growing cache (beam search without compression) reuses the packed records and rewrites only the sizes
    recs = slab._reorder_recs
    slab.lengths = [6, 1, 16]
    regions = unpack(slab._reorder_records())
    assert slab._reorder_recs is recs
    assert [r[3] for r in regions] == [6 * D * e, 6 * D * e, 6 * e, D * e, D * e, e, 16 * D * e, 16 * D * e, 16 * e]
    assert [r[:3] for r in regions][0] == k0[:3]


def test_follower_records_describe_their_live_buffers():
    win = SnapKVQueryWindow(2, 4, 6, 64, 8, torch.bfloat16, device="cpu")
    win.filled = [3, 0]
    r0, r1 = unpack(win._reorder_records(4, torch.device("cpu")))
    assert r0 == (win.queries[0].data_ptr(), 6 * 8 * 64 * 2, 8 * 64 * 2, 3 * 64 * 2, 6, 2)
    assert r1[0] == win.queries[1].data_ptr() and r1[3] == 0
    # a window of another shape (it may reuse a freed window's address): its records describe its own strides
    small = SnapKVQueryWindow(2, 4, 6, 64, 4, torch.bfloat16, device="cpu")
    small.filled = [3, 0]
    s0 = unpack(small._reorder_records(4, torch.device("cpu")))[0]
    assert s0[1:3] == (6 * 4 * 64 * 2, 4 * 64 * 2) and s0[1:3] != r0[1:3]

    h2o = H2OScoreSlab(num_layers=2, capacity=32)
    assert h2o._reorder_records(4, torch.device("cpu")) == b""        # no buffers yet: nothing moves
    h2o._ensure(4, 8, torch.float32, torch.device("cpu"), 32)
    h2o._lens = {1: 7}
    h2o._scored = {1: (4, 5)}
    a0, a1 = unpack(h2o._reorder_records(4, torch.device("cpu")))
    assert a0[3] == 0 and a1 == (h2o._acc[1].data_ptr(), 8 * 32 * 4, 32 * 4, 7 * 4, 8, 4)
    assert h2o._scored == {}                                          # score rows are rebuilt after a reorder
    # the accumulators are reallocated (a longer key_len doubles the capacity): new pointers and strides
    h2o._ensure(4, 8, torch.float32, torch.device("cpu"), 40)
    h2o._lens = {1: 40}
    b1 = unpack(h2o._reorder_records(4, torch.device("cpu")))[1]
    assert b1 == (h2o._acc[1].data_ptr(), 8 * 64 * 4, 64 * 4, 40 * 4, 8, 4)


def test_index_checks():
    dev = torch.device("cpu")
    with pytest.raises(ValueError):
        _engine.reorder_index(torch.tensor([0, 1, 2]), 4, dev)             # wrong length
    with pytest.raises(ValueError):
        _engine.reorder_index([0, 1], 4, dev)
    with pytest.raises(ValueError):
        _engine.reorder_index(torch.tensor([0.0, 1.0, 2.0, 3.0]), 4, dev)  # float
    with pytest.raises(ValueError):
        _engine.reorder_index(torch.zeros((2, 2), dtype=torch.int64), 4, dev)  # 2-D
    with pytest.raises(ValueError):
        _engine.reorder_index(torch.tensor([0, 1, 4, 3]), 4, dev)          # out of range on the host
    with pytest.raises(ValueError):
        _engine.reorder_index([0, -1, 2, 3], 4, dev)
    with pytest.raises(ValueError):
        _engine.reorder_index([0.5, 1, 2, 3], 4, dev)
    got = _engine.reorder_index([3, 3, 0, 1], 4, dev)
    assert got.dtype == torch.int64 and got.tolist() == [3, 3, 0, 1]


def test_pinned_slab_and_follower_batch_are_refused():
    with pytest.raises(ValueError, match="pinned"):
        host_slab(pinned=True).reorder_([0, 1, 2, 3])
    slab = host_slab(B=4)
    with pytest.raises(ValueError, match="batch"):
        slab.reorder_([0, 1, 2, 3], SnapKVQueryWindow(1, 2, 2, 64, 4, torch.bfloat16, device="cpu"))
    h2o = H2OScoreSlab(num_layers=3)
    h2o._ensure(2, 2, torch.float16, torch.device("cpu"), 16)
    h2o._lens = {0: 3}
    with pytest.raises(ValueError, match="batch"):
        h2o._reorder_records(4, torch.device("cpu"))


def test_abi_refusals():
    lib = _engine.load_library()
    buf = (ctypes.c_int64 * 64)()
    p = ctypes.addressof(buf)
    idx = (ctypes.c_int64 * 4)(0, 0, 1, 1)

    def region(base=p, sb=64, su=16, ub=16, units=2, e=2):
        return _engine.pack_regions([(base, sb, su, ub, units, e)])

    def call(batch=4, index=ctypes.addressof(idx), bits=64, n=1, recs=None):
        return lib.kvc_batch_reorder(0, batch, index, bits, n, region() if recs is None else recs, None)

    assert call(n=0, recs=b"") == 0
    assert call(recs=region(units=0)) == 0                 # nothing to move: no launch, no CUDA call
    assert call(index=None) == INVALID
    assert call(batch=0) == INVALID and call(batch=1025) == INVALID
    assert call(bits=16) == INVALID
    assert lib.kvc_batch_reorder(0, 4, ctypes.addressof(idx), 64, 1, None, None) == INVALID
    assert call(recs=region(base=0)) == INVALID             # NULL base
    assert call(recs=region(ub=-2)) == INVALID and call(recs=region(units=-1)) == INVALID
    assert call(recs=region(sb=-64)) == INVALID
    assert call(recs=region(sb=16, su=16)) == INVALID      # batch entries overlap
    assert call(recs=region(su=8)) == INVALID              # units of one entry overlap
    assert call(recs=region(base=p + 1)) == UNSUPPORTED    # misaligned for 2-byte elements
    assert call(recs=region(ub=6, e=4)) == UNSUPPORTED
    assert call(recs=region(sb=66, e=4)) == UNSUPPORTED    # a stride that is not a multiple of elem_bytes
    assert call(recs=region(e=3)) == UNSUPPORTED
