"""The library's host decisions, pinned without a GPU: the status every compaction and vote entry point returns for
arguments refused before any CUDA call, and what the planning queries (kvc_workspace_bytes, kvc_launch_shape) answer.

Every expected value was recorded from the library before its host code was restructured; the two compaction forms
share their plan checks, chunk summary and launch planning, and these tables hold them to the same answers.  Pointers
are fake (aligned or not, never dereferenced): every argument set below fails validation, so no case reaches the
device."""

import ctypes
import json
import os

import pytest

from kvcompress import _engine
from kvcompress import _planner as P
from kvcompress.slab_cache import _SLAB

F32, F16, BF16 = 0, 1, 2
INVALID, UNSUPPORTED, TOO_LARGE = 1, 2, 3
A = 0x100000  # a 16-byte aligned fake device address


def _plan(S=1000, sink=4, lo=4, hi=900, k=64, tail=100, score=P.SCORE_L2_LOW, pool=1):
    return _engine._PLAN.pack(S, sink, lo, hi, k, tail, score, pool)


def _io(k_in=A, v_in=A, k_out=A, v_out=A, ks=(64000, 64000, 64), vs=(64000, 64000, 64), idx_in=0, score_in=0):
    return _engine._IO.pack(k_in, v_in, k_out, v_out, *ks, *vs, 0, idx_in, score_in, 0, 0, 0)


def _slab(k=A, v=A, norms=A, ks=(64000, 64000), vs=(64000, 64000)):
    return _SLAB.pack(k, v, norms, *ks, *vs, 1000, 1000)


def _carry(acc=A, group=2, prev_len=900):
    return _engine._CARRY.pack(acc, 8000, 1000, group, prev_len)


def _vote(k=A, q=A, votes=A, ks=(64000, 64000, 64), qs=(4096, 2048, 64), S=1000):
    return _engine._VOTE.pack(k, q, votes, *ks, *qs, S, 0, 0)


def _shape(dtype=BF16, D=64, B=2, H=4):
    return _engine._SHAPE.pack(B, H, D, dtype, 0)


GOOD = _plan()


def _case(plans, io=None, slabs=None, carry=None, shape=None, forms="fs"):
    """forms: the compaction forms the case applies to, f = out of place (kvc_compress_layers*), s = in place
    (kvc_slab_compress*).  A plan that breaks only the in-place rule is valid out of place, so it is an "s" case."""
    n = len(plans)
    return dict(plans=b"".join(plans), n=n, io=b"".join(io or [_io()] * n), slabs=b"".join(slabs or [_slab()] * n),
                carry=b"".join(carry) if carry else None, shape=shape or _shape(), forms=forms)


COMPACTION = {
    "neg_seq_len": _case([_plan(S=-1)]),
    "sink_past_end": _case([_plan(sink=1001)]),
    "tail_past_end": _case([_plan(tail=1001)]),
    "sel_lo_negative": _case([_plan(lo=-1)]),
    "sel_hi_past_end": _case([_plan(hi=1001)]),
    "sel_lo_above_hi": _case([_plan(lo=500, hi=400)]),
    "k_sel_over_region": _case([_plan(lo=4, hi=50, k=47)]),
    "score_none_with_select": _case([_plan(score=P.SCORE_NONE)]),
    "score_out_of_range": _case([_plan(score=7)]),
    "given_index_no_rows": _case([_plan(score=P.SCORE_GIVEN_INDEX)]),
    "given_score_no_scores": _case([_plan(score=P.SCORE_GIVEN_SCORE)]),
    "shared_score_no_scores": _case([_plan(score=P.SCORE_GIVEN_SCORE_SHARED)]),
    "pool_too_wide": _case([_plan(score=P.SCORE_SNAPKV_POOL, pool=65)]),
    "no_scores_and_pool_too_wide": _case([_plan(score=P.SCORE_GIVEN_SCORE, pool=65)]),
    "C_over_S": _case([_plan(sink=400, tail=600)], forms="s"),
    "region_into_sinks": _case([_plan(sink=10, lo=4)], forms="s"),
    "region_into_tail": _case([_plan(hi=950)], forms="s"),
    "region_into_tail_and_pool_too_wide": _case([_plan(hi=950, score=P.SCORE_SNAPKV_POOL, pool=65)]),
    "layer1_bad_behind_layer0": _case([GOOD, _plan(k=900)]),
    "layer1_pool_behind_layer0": _case([GOOD, _plan(score=P.SCORE_SNAPKV_POOL, pool=65)]),
    "null_k_in": _case([GOOD], [_io(k_in=0)], [_slab(k=0)]),
    "null_out": _case([GOOD], [_io(v_out=0)], [_slab(norms=0)]),
    "misaligned_rows": _case([GOOD], [_io(v_in=A + 8)], [_slab(v=A + 8)]),
    "misaligned_stride": _case([GOOD], [_io(ks=(64000, 64000, 68))], [_slab(ks=(64004, 64000))]),
    "null_k_in_and_pool_too_wide": _case([_plan(score=P.SCORE_SNAPKV_POOL, pool=65)], [_io(k_in=0)], [_slab(k=0)]),
    "rows_too_large": _case([_plan(S=1 << 30, sink=0, lo=0, hi=0, k=0, tail=1 << 30)], forms="f"),
    "carry_group_0": _case([GOOD], carry=[_carry(group=0)]),
    "carry_prev_negative": _case([GOOD], carry=[_carry(prev_len=-1)]),
    "carry_misaligned": _case([GOOD], carry=[_carry(acc=A + 1)]),
    "carry_not_in_place": _case([_plan(hi=950)], carry=[_carry()]),
    "carry_not_in_place_and_pool_too_wide": _case([_plan(hi=950, score=P.SCORE_SNAPKV_POOL, pool=65)],
                                                  carry=[_carry()]),
    "carry_layer1_behind_layer0": _case([GOOD, GOOD], carry=[_carry(acc=0, group=0), _carry(group=0)]),
    "dtype_unknown": _case([GOOD], shape=_shape(dtype=3)),
    "row_not_16B": _case([GOOD], shape=_shape(D=36)),
    "row_over_2KB": _case([GOOD], shape=_shape(D=2048)),
    "batch_zero": _case([GOOD], shape=_shape(B=0)),
}


def _compaction_statuses(c):
    """[kvc_compress_layers, kvc_compress_layers_carry, kvc_slab_compress, kvc_slab_compress_carry] statuses of the
    case (the plain entry points only without a carry; the forms the case does not apply to are left out)."""
    lib = _engine.load_library()
    n, shape, plans, carry = c["n"], c["shape"], c["plans"], c["carry"]
    idx_in = (ctypes.c_void_p * n)()  # no caller rows or scores for any layer
    got = []
    if "f" in c["forms"]:
        if carry is None:
            got.append(lib.kvc_compress_layers(shape, n, plans, c["io"], None))
        got.append(lib.kvc_compress_layers_carry(shape, n, plans, c["io"], carry, None, 0, None))
    if "s" in c["forms"]:
        if carry is None:
            got.append(lib.kvc_slab_compress(shape, n, plans, c["slabs"], None, idx_in, None, 0, None))
        got.append(lib.kvc_slab_compress_carry(shape, n, plans, c["slabs"], None, idx_in, carry, None, 0, None))
    return got


VOTE_PLAN = _plan(S=1000, sink=0, lo=0, hi=968, k=200, tail=32, score=P.SCORE_GIVEN_SCORE, pool=5)

# name -> (vote records, plans, io records, shape, group, window)
VOTE = {
    "f32": ([_vote()], None, None, _shape(dtype=F32, D=32)),
    "row_width_96": ([_vote()], None, None, _shape(D=96)),
    "group_window_over_M": ([_vote()], None, None, None, 4, 64),
    "group_zero": ([_vote()], None, None, None, 0),
    "window_zero": ([_vote()], None, None, None, 2, 0),
    "null_q": ([_vote(q=0)],),
    "seq_len_not_past_window": ([_vote(S=32)],),
    "misaligned_keys": ([_vote(k=A + 8)],),
    "misaligned_query_stride": ([_vote(qs=(4096, 2048, 68))],),
    "layer1_bad_behind_layer0": ([_vote(), _vote(votes=0)],),
    "plan_with_sinks": ([_vote()], [_plan(S=1000, sink=4, lo=0, hi=968, k=200, tail=32, score=P.SCORE_GIVEN_SCORE)]),
    "plan_not_given_score": ([_vote()], [_plan(S=1000, sink=0, lo=0, hi=968, k=200, tail=32)]),
    "plan_pool_too_wide": ([_vote()], [_plan(S=1000, sink=0, lo=0, hi=968, k=200, tail=32,
                                             score=P.SCORE_GIVEN_SCORE, pool=65)]),
    "null_q_and_plan_pool_too_wide": ([_vote(q=0)], [_plan(S=1000, sink=0, lo=0, hi=968, k=200, tail=32,
                                                            score=P.SCORE_GIVEN_SCORE, pool=65)]),
    "io_keys_differ": ([_vote()], [VOTE_PLAN], [_io(k_in=A + 16)]),
    "io_values_misaligned": ([_vote()], [VOTE_PLAN], [_io(v_out=A + 8)]),
    "io_key_strides_differ": ([_vote()], [VOTE_PLAN], [_io(ks=(64000, 64000, 128))]),
    "prefix_too_large": ([_vote(S=1 << 20)], [_plan(S=1 << 20, sink=0, lo=0, hi=(1 << 20) - 32, k=200, tail=32,
                                                     score=P.SCORE_GIVEN_SCORE)]),
    "plan_layer1_behind_layer0": ([_vote(), _vote()], [VOTE_PLAN, _plan(S=1000, sink=0, lo=0, hi=968, k=0, tail=32,
                                                                         score=P.SCORE_GIVEN_SCORE)]),
}


def _vote_statuses(case):
    votes, plans, io, shape, group, window = (list(case) + [None] * 6)[:6]
    n = len(votes)
    shape = shape or _shape()
    group = 2 if group is None else group
    window = 32 if window is None else window
    plans = plans or [VOTE_PLAN] * n
    io = io or [_io()] * n
    lib = _engine.load_library()
    v_b = b"".join(votes)
    return [lib.kvc_snapkv_vote(shape, n, v_b, group, window, None) if len(case) == 1 or case[1] is None else None,
            lib.kvc_snapkv_vote_compress(shape, n, v_b, b"".join(plans), b"".join(io), group, window, None)]


def _planner_plans():
    """GATHER plans of every planner: short and long layers, and a 200K-row region that needs the workspace."""
    lens = [1000, 4096, 4096, 9000]
    sets = {
        "l2": P.plan_l2(lens, 0.5, 512, []),
        "fix_size_low": P.plan_fix_size(lens, 2048, 0.5, "keep_low", []),
        "fix_size_high": P.plan_fix_size(lens, 2048, 0.5, "keep_high", []),
        "fix_size_random": P.plan_fix_size(lens, 2048, 0.5, "random", []),
        "streaming": P.plan_streaming(lens, 4, 1020, []),
        "evict_for_space": P.plan_evict_for_space(lens, 64, 4, 2000, []),
        "h2o": P.plan_h2o(lens, 4, 256, 764, []),
        "h2o_given_score": P.plan_h2o(lens, 4, 256, 764, [], score=P.SCORE_GIVEN_SCORE),
        "snapkv": P.plan_snapkv(lens, 32, 1024, 5, []),
        "pyramid": P.plan_pyramid(lens, 1024, 0.9, 128, "pyramid", []),
        "adaptive": P.plan_adaptive(lens, 2048, 3000, 6000, 0.3, 0.8, []),
        "recent_only": P.plan_recent_only(lens, 1024, []),
        "h2o_200k": P.plan_h2o([200_000], 4, 4096, 1020, []),
        "snapkv_200k": P.plan_snapkv([200_000], 32, 8192, 7, []),
    }
    out = {}
    for name, plans in sets.items():
        g = [p for p in plans if p.kind == P.GATHER]
        out[name] = b"".join(_engine._PLAN.pack(p.seq_len, p.sink, p.sel_lo, p.sel_hi, p.k_sel, p.tail, p.score,
                                                p.pool_kernel) for p in g), len(g)
    return out


BH = [(1, 1), (1, 8), (4, 16), (32, 32)]


def _planner_answers():
    lib = _engine.load_library()
    got = {}  # "planner/dtype/head_dim" -> [workspace bytes, launch_shape status, nt, ctas, nsw, ws] per B x H
    for name, (plan_b, n) in _planner_plans().items():
        for dtype in (F32, F16, BF16):
            for D in (64, 80, 96, 128):
                rows = got[f"{name}/{dtype}/{D}"] = []
                for B, H in BH:
                    shape = _shape(dtype=dtype, D=D, B=B, H=H)
                    out = (ctypes.c_int32 * 4)()
                    st = lib.kvc_launch_shape(shape, n, plan_b, out)
                    rows.append([int(lib.kvc_workspace_bytes(shape, n, plan_b)), st, *out])
    return got


_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host_checks.json")


def _golden():
    with open(_GOLDEN) as f:
        return json.load(f)


@pytest.mark.parametrize("name", sorted(COMPACTION))
def test_compaction_status(name):
    got = _compaction_statuses(COMPACTION[name])
    assert got and all(s in (INVALID, UNSUPPORTED, TOO_LARGE) for s in got)  # refused before any CUDA call
    assert got == _golden()["compaction"][name]


@pytest.mark.parametrize("name", sorted(VOTE))
def test_vote_status(name):
    got = [s for s in _vote_statuses(VOTE[name]) if s is not None]
    assert got and all(s in (INVALID, UNSUPPORTED, TOO_LARGE) for s in got)  # refused before any CUDA call
    assert got == _golden()["vote"][name]


def test_planner_answers():
    """kvc_workspace_bytes and kvc_launch_shape over every planner, three dtypes, head_dim 64/80/96/128 and B*H from
    1 to 1024."""
    want = _golden()["planner"]
    got = _planner_answers()
    assert sorted(got) == sorted(want)
    bad = {k: (got[k], want[k]) for k in want if got[k] != want[k]}
    assert not bad, dict(list(bad.items())[:10])
    rows = [r for v in want.values() for r in v]
    assert any(r[0] > 0 for r in rows) and any(r[5] == 1 for r in rows)  # the workspace path is covered
