"""H2OScoreSlab without a GPU: the C ABI of kvc_h2o_accumulate (argument checks, struct layout) and the host
arithmetic that turns accumulator lengths into compaction plans (reference h2o_attention.py:153-213, :318-331)."""

import ctypes

import pytest
import torch

import kvcompress
from kvcompress import _engine
from kvcompress import _planner as P
from kvcompress.methods._common import cached_plans
from kvcompress.slab_cache import _SLAB


def _layer(attn=16, acc=16, score=16, n_query=1, key_len=100, prev_len=-1, lo=4, hi=50):
    return _engine._H2O.pack(attn, 100, 100, 100, acc, 128, 128, score, n_query, key_len, prev_len, lo, hi, 0)


def test_accumulate_struct_matches_the_header():
    assert _engine._H2O.size == 88
    assert P.SCORE_GIVEN_SCORE_SHARED == 6


def test_accumulate_argument_checks():
    """Validation happens before any CUDA call, so it is testable without a GPU."""
    lib = _engine.load_library()
    stream = ctypes.c_void_p(0)
    bf16 = _engine._SHAPE.pack(1, 4, 0, 2, 0)
    assert lib.kvc_h2o_accumulate(bf16, 1, None, 0.9, stream) == 1                          # null layers
    assert lib.kvc_h2o_accumulate(None, 1, _layer(), 0.9, stream) == 1                      # null shape
    assert lib.kvc_h2o_accumulate(bf16, 1, _layer(hi=101), 0.9, stream) == 1                # score_hi > key_len
    assert lib.kvc_h2o_accumulate(bf16, 1, _layer(lo=60, hi=50), 0.9, stream) == 1          # score_lo > score_hi
    assert lib.kvc_h2o_accumulate(bf16, 1, _layer(acc=0), 0.9, stream) == 1                 # no accumulators
    assert lib.kvc_h2o_accumulate(bf16, 1, _layer(score=0), 0.9, stream) == 1               # score region, no output
    assert lib.kvc_h2o_accumulate(bf16, 1, _layer(n_query=0), 0.9, stream) == 1             # attention of 0 queries
    assert lib.kvc_h2o_accumulate(_engine._SHAPE.pack(0, 4, 0, 2, 0), 1, _layer(), 0.9, stream) == 1
    assert lib.kvc_h2o_accumulate(_engine._SHAPE.pack(1, 4, 0, 7, 0), 1, _layer(), 0.9, stream) == 2  # bad dtype
    assert lib.kvc_h2o_accumulate(bf16, 1, _layer(attn=17), 0.9, stream) == 2               # misaligned element
    assert lib.kvc_h2o_accumulate(bf16, 0, None, 0.9, stream) == 0                          # nothing to do


def test_shared_score_plans_are_validated():
    """KVC_SCORE_GIVEN_SCORE_SHARED needs its score row like GIVEN_SCORE; kinds past it are refused."""
    lib = _engine.load_library()
    shape = _engine._SHAPE.pack(1, 1, 16, 2, 0)
    io = _engine._IO.pack(16, 16, 16, 16, 160, 160, 16, 160, 160, 16, 0, 0, 0, 0, 0, 0)
    no_scores = _engine._PLAN.pack(10, 1, 1, 9, 3, 1, P.SCORE_GIVEN_SCORE_SHARED, 1)
    assert lib.kvc_compress_layers(shape, 1, no_scores, io, None) == 1
    past_last = _engine._PLAN.pack(10, 1, 1, 9, 3, 1, 7, 1)
    assert lib.kvc_compress_layers(shape, 1, past_last, io, None) == 1
    slab = _SLAB.pack(16, 16, 16, 160, 160, 160, 160, 16, 16)
    assert lib.kvc_slab_compress(shape, 1, no_scores, slab, None, None, None, 0, None) == 1


@pytest.mark.parametrize("seq_len,acc_len,want", [
    (700, 700, (4, 608, 32)),     # the update's own region
    (700, 500, (4, 408, 32)),     # accumulators shorter than the cache: acc_len bounds the region
    (129, 700, (4, 37, 32)),      # accumulators longer than the cache: the cache bounds it
    (120, 120, (4, 28, 24)),      # fewer rows than heavy hitters: all of them
    (96, 96, (0, 0, 0)),          # empty middle
    (700, 90, (0, 0, 0)),         # empty middle through a short accumulator
])
def test_score_region_arithmetic(seq_len, acc_len, want):
    assert P.h2o_score_region(seq_len, acc_len, 4, 32, 92) == want


class _Recorder:
    """Stands in for the re-scoring launch: records the layers and marks their rows as scored."""

    def __init__(self, manager):
        self.manager, self.calls = manager, []

    def __call__(self, layers):
        self.calls.append(list(layers))
        for li, lo, hi in layers:
            self.manager._scored[li] = (lo, hi)


def _fake_manager(lens, scored, B=2, Hq=4, cap=1024, dtype=torch.bfloat16):
    """An H2OScoreSlab whose buffers live on the CPU: the compaction planning never touches their contents."""
    m = kvcompress.H2OScoreSlab(start_size=4, heavy_hitter_size=32, recent_size=92, num_layers=len(lens), num_heads=Hq)
    m._acc = torch.zeros((len(lens), B, Hq, cap), dtype=dtype)
    m._score = torch.zeros((len(lens), B, cap), dtype=dtype)
    m._lens = {li: n for li, n in enumerate(lens) if n is not None}
    m._scored = dict(scored)
    m._rescore = _Recorder(m)
    return m


def test_compress_plans_from_accumulator_lengths():
    """Per layer: scores over [start, min(S, acc_len) - recent) with count = min(hh, region); a region other than the
    one last scored is re-scored (one call for all such layers); no data -> evenly spaced rows; empty -> no heavy
    hitter; skipped layers untouched."""
    S = 700
    lens = [None, 700, 500, 900, 90, 700]
    scored = {1: (4, 608), 2: (4, 408), 3: (4, 808), 4: (0, 0), 5: (4, 608)}
    m = _fake_manager(lens, scored)
    plans = cached_plans(P.plan_h2o, [S] * len(lens), 4, 32, 92, skip_layers=(5,))
    ps, given, scores = m.compress_plans(plans, 4, 32, 92, 2, 3, torch.bfloat16, "cpu")
    # layer 3's accumulators cover 900 keys, the cache 700 rows: its row must be re-scored over [4, 608)
    assert m._rescore.calls == [[(3, 4, 608)]]
    p0, p1, p2, p3, p4, p5 = ps.plans
    assert (p0.score, p0.k_sel, p0.sel_lo, p0.sel_hi) == (P.SCORE_GIVEN_INDEX, 32, 4, 608)
    step = (S - 92 - 4) // 32
    assert given[0].shape == (2, 3, 32) and given[0].dtype == torch.int32
    assert given[0][1, 2].tolist() == [4 + step * i for i in range(32)]
    assert (p1.score, p1.k_sel, p1.sel_lo, p1.sel_hi, p1.sink, p1.tail) == (P.SCORE_GIVEN_SCORE_SHARED, 32, 4, 608, 4, 92)
    assert (p2.score, p2.k_sel, p2.sel_hi) == (P.SCORE_GIVEN_SCORE_SHARED, 32, 408)   # acc_len < S
    assert (p3.score, p3.k_sel, p3.sel_hi) == (P.SCORE_GIVEN_SCORE_SHARED, 32, 608)   # acc_len > S
    assert (p4.score, p4.k_sel, p4.out_len) == (P.SCORE_NONE, 0, 96)                  # empty middle
    assert p5.kind == P.KEEP
    assert set(scores) == {1, 2, 3} and scores[2].shape == (2, 404) and scores[1].shape == (2, 604)
    assert scores[1].data_ptr() == m._score[1].data_ptr()                              # a view of the score buffer
    assert [p.out_len for p in ps.plans] == [128, 128, 128, 128, 96, 700]
    # the same decision again: the cached plan set, no re-score (the row now holds the compaction's region)
    ps2, _, _ = m.compress_plans(plans, 4, 32, 92, 2, 3, torch.bfloat16, "cpu")
    assert ps2 is ps and len(m._rescore.calls) == 1


def test_compress_plans_refuse_mismatches():
    m = _fake_manager([700], {0: (4, 608)})
    plans = cached_plans(P.plan_h2o, [700], 4, 32, 92, skip_layers=())
    with pytest.raises(ValueError, match="bfloat16.*float16|float16.*bfloat16"):
        m.compress_plans(plans, 4, 32, 92, 2, 3, torch.float16, "cpu")
    with pytest.raises(ValueError, match="batch"):
        m.compress_plans(plans, 4, 32, 92, 5, 3, torch.bfloat16, "cpu")
    other = cached_plans(P.plan_h2o, [700], 4, 16, 92, skip_layers=())
    with pytest.raises(ValueError, match="same sizes"):
        m.compress_plans(other, 4, 16, 92, 2, 3, torch.bfloat16, "cpu")


def test_reset_and_views_are_host_only():
    m = _fake_manager([700, None], {0: (4, 608)})
    acc = m.accumulated_attention
    assert list(acc) == [0] and 1 not in acc and acc[0].shape == (2, 4, 700)
    assert acc[0].data_ptr() == m._acc.data_ptr()
    m.current_seq_len = 700
    m.reset()
    assert len(m.accumulated_attention) == 0 and m.current_seq_len == 0
    assert m._acc is not None  # the buffers stay allocated


def test_exports():
    from kvcompress import methods

    assert kvcompress.H2OScoreSlab is methods.H2OScoreSlab
    assert "H2OScoreSlab" in kvcompress.__all__ and "H2OScoreSlab" in methods.__all__
