"""Cumulative H2O without a GPU: the C ABI of kvc_slab_compress_carry / kvc_compress_layers_carry (struct layout,
exported symbols, argument checks that run before any CUDA call) and the refusals of carry_scores=True with the torch
manager."""

import ctypes

import pytest
import torch

import kvcompress
from kvcompress import H2OAttentionManager, H2OScoreSlab, KVSlabCache, _engine
from kvcompress import _planner as P
from kvcompress.slab_cache import _SLAB

BF16, F32 = 2, 0


class _CarryLayer(ctypes.Structure):
    """kvc_carry_layer as include/kvc.h declares it."""
    _fields_ = [("acc", ctypes.c_void_p), ("acc_stride_b", ctypes.c_int64), ("acc_stride_h", ctypes.c_int64),
                ("group", ctypes.c_int32), ("prev_len", ctypes.c_int32)]


def test_carry_struct_matches_the_header():
    assert ctypes.sizeof(_CarryLayer) == 32 == _engine._CARRY.size
    rec = _engine._CARRY.pack(0x1000, 3, 5, 4, 77)
    c = _CarryLayer.from_buffer_copy(rec)
    assert (c.acc, c.acc_stride_b, c.acc_stride_h, c.group, c.prev_len) == (0x1000, 3, 5, 4, 77)


def test_both_entry_points_are_exported():
    lib = ctypes.CDLL(_engine.library_path())
    assert hasattr(lib, "kvc_slab_compress_carry") and hasattr(lib, "kvc_compress_layers_carry")
    assert _engine.load_library().kvc_abi_version() == 5


def _carry(acc=0x1000, group=2, prev_len=10):
    return _engine._CARRY.pack(acc, 4096, 512, group, prev_len)


def _calls(dtype, carry, plan=None):
    """Status of both entry points on a 1 x 1 layer (S 10: sink 1, 3 of [1, 9), tail 1) with the given carry record.
    Pointers are fake: a status other than KVC_ERR_INVALID_ARG would have meant reaching the device."""
    lib = _engine.load_library()
    D = 16 if dtype == F32 else 32
    shape = _engine._SHAPE.pack(1, 1, D, dtype, 0)
    plan = plan or _engine._PLAN.pack(10, 1, 1, 9, 3, 1, P.SCORE_GIVEN_INDEX, 1)
    io = _engine._IO.pack(16, 16, 16, 16, 160, 160, 16, 160, 160, 16, 0, 16, 0, 0, 0, 0)
    slab = _SLAB.pack(16, 16, 16, 160, 160, 160, 160, 16, 16)
    idx_in = (ctypes.c_void_p * 1)(16)
    a = lib.kvc_compress_layers_carry(shape, 1, plan, io, carry, None, 0, None)
    b = lib.kvc_slab_compress_carry(shape, 1, plan, slab, None, idx_in, carry, None, 0, None)
    return a, b


@pytest.mark.parametrize("dtype", [F32, BF16])
def test_carry_argument_checks(dtype):
    """KVC_ERR_INVALID_ARG before any CUDA call: group < 1, prev_len < 0, acc rows not aligned to the element size;
    a carried layer must also be a valid in-place compaction (C <= S, the region between the sinks and the tail)."""
    assert _calls(dtype, _carry(group=0)) == (1, 1)
    assert _calls(dtype, _carry(group=-3)) == (1, 1)
    assert _calls(dtype, _carry(prev_len=-1)) == (1, 1)
    assert _calls(dtype, _carry(acc=0x1001)) == (1, 1)          # odd address: misaligned for every dtype
    if dtype == F32:
        assert _calls(dtype, _carry(acc=0x1002)) == (1, 1)      # 2-byte aligned is not enough for fp32
    overlap = _engine._PLAN.pack(10, 4, 0, 10, 3, 4, P.SCORE_GIVEN_INDEX, 1)   # region reaches into the sinks / tail
    assert _calls(dtype, _carry(), overlap)[0] == 1
    too_many = _engine._PLAN.pack(10, 5, 0, 0, 0, 6, P.SCORE_NONE, 1)         # C = 11 > S
    assert _calls(dtype, _carry(), too_many)[0] == 1


def test_carry_checks_skip_layers_without_acc():
    """acc == NULL: the layer carries nothing, so its other carry fields are not looked at (the plain entry point's
    own checks still apply, as a bad plan shows)."""
    bad_plan = _engine._PLAN.pack(10, 1, 1, 9, 11, 1, P.SCORE_GIVEN_INDEX, 1)  # k_sel > region
    assert _calls(F32, _carry(acc=0, group=0, prev_len=-5), bad_plan) == (1, 1)
    assert _calls(F32, None, bad_plan) == (1, 1)


def test_carry_record_validation():
    """The Python side refuses what the library would, and host tensors: the carried state lives on the device."""
    acc = torch.zeros(2, 8, 64)
    with pytest.raises(ValueError, match="CUDA"):
        _engine.carry_record(3, (acc, 4, 40), 2, 2, torch.float32, 50)     # host memory
    with pytest.raises(ValueError, match="group"):
        _engine.carry_record(3, (acc, 0, 40), 2, 2, torch.float32, 50)     # group < 1
    with pytest.raises(ValueError, match="prev_len"):
        _engine.carry_record(3, (acc, 4, -1), 2, 2, torch.float32, 50)     # prev_len < 0


def test_carry_scores_refuses_the_torch_manager():
    """carry_scores=True needs H2OScoreSlab(carry_scores=True): in the harness, the function and compress_."""
    from kvcompress.evaluate_attention import evaluate_with_attention_compression

    model = torch.nn.Linear(2, 2)
    ids = torch.zeros(1, 8, dtype=torch.long)
    for manager in (H2OAttentionManager(), H2OScoreSlab()):
        with pytest.raises(ValueError, match="carry_scores"):
            evaluate_with_attention_compression(model, h2o_manager=manager, carry_scores=True, input_ids=ids,
                                                show_progress=False)
    kv = [(torch.zeros(1, 2, 8, 16), torch.zeros(1, 2, 8, 16))]
    with pytest.raises(ValueError, match="carry_scores"):
        kvcompress.h2o_attention_compress(kv, h2o_manager=H2OAttentionManager(), carry_scores=True)
    with pytest.raises(ValueError, match="carry_scores"):
        kvcompress.h2o_attention_compress(kv, h2o_manager=H2OScoreSlab(carry_scores=True), carry_scores=False)
    # the slab's in-place form checks before it touches the cache (no GPU needed to get there)
    slab = object.__new__(KVSlabCache)
    with pytest.raises(ValueError, match="carry_scores"):
        slab.compress_("h2o_attention", h2o_manager=H2OAttentionManager(), carry_scores=True)


def test_carry_scores_default_is_off():
    assert H2OScoreSlab().carry_scores is False
    assert H2OScoreSlab(carry_scores=True).carry_scores is True
