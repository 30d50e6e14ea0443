"""The tensor-core H2O query update without a GPU: the C ABI of kvc_h2o_accumulate_qk_tc (exported symbols, refusals
that run before any CUDA call, workspace arithmetic) and the ValueErrors of H2OScoreSlab(tensor_cores=True)."""

import ctypes

import pytest
import torch

from kvcompress import H2OScoreSlab, _engine

F32, F16, BF16 = 0, 1, 2


def _shape(B=1, H=2, D=128, dt=BF16):
    return _engine._SHAPE.pack(B, H, D, dt, 0)


def _layer(q=1024, k=1024, mask=0, acc=16, score=16, n_query=1, key_len=100, prev_len=-1, lo=4, hi=50, ks=128,
           qs=(8192, 1024, 128), scaling=0.088):
    return _engine._H2O_QK.pack(q, qs[0], qs[1], qs[2], k, ks * 200, ks * 100, ks, mask, 1000, 100, acc, 800, 200, score,
                                scaling, n_query, key_len, prev_len, lo, hi)


def _lib():
    return _engine.load_library()


def _ws(shape, group, recs, n=1):
    return _lib().kvc_h2o_qk_tc_workspace_bytes(shape, group, n, recs)


def _run(shape, group, recs, n=1, ws=1 << 20, ws_bytes=1 << 20):
    return _lib().kvc_h2o_accumulate_qk_tc(shape, group, n, recs, 0.9, ctypes.c_void_p(ws), ws_bytes, None)


def test_symbols_are_exported():
    lib = ctypes.CDLL(_engine.library_path())
    for name in ("kvc_h2o_accumulate_qk_tc", "kvc_h2o_qk_tc_workspace_bytes"):
        assert hasattr(lib, name), name
    assert lib.kvc_abi_version() == 5


def test_everything_the_cuda_core_form_refuses_is_refused():
    s = _shape()
    assert _run(None, 2, _layer()) == 1                                    # null shape
    assert _run(s, 2, None) == 1                                           # null layers
    assert _run(s, 0, _layer()) == 1                                       # group < 1
    assert _run(s, 2, _layer(n_query=101)) == 1                            # more queries than keys, no mask
    assert _run(s, 2, _layer(hi=101)) == 1                                 # score region beyond key_len
    assert _run(s, 2, _layer(lo=-1)) == 1                                  # score region before 0
    assert _run(s, 2, _layer(lo=60, hi=50)) == 1                           # score_lo > score_hi
    assert _run(s, 2, _layer(score=0)) == 1                                # score region, no output
    assert _run(s, 2, _layer(acc=0)) == 1                                  # no accumulators
    assert _run(s, 2, _layer(q=0)) == 1                                    # no queries
    assert _run(s, 2, _layer(k=0)) == 1                                    # no keys
    assert _run(s, 2, _layer(n_query=0)) == 1                              # no queries
    assert _run(_shape(B=0), 2, _layer()) == 1
    need = _ws(s, 2, _layer())
    assert need > 0
    assert _run(s, 2, _layer(), ws=0, ws_bytes=0) == 1                     # no workspace
    assert _run(s, 2, _layer(), ws_bytes=need - 1) == 1                    # workspace too small
    assert _run(s, 2, _layer(), ws=1 << 20 | 8) == 1                       # workspace not 16-byte aligned
    assert _run(_shape(dt=7), 2, _layer()) == 2                            # dtype
    assert _run(_shape(), 2, _layer(k=24)) == 2                            # K not 16-byte aligned
    assert _run(_shape(), 2, _layer(ks=60)) == 2                           # K row stride not 16-byte aligned
    assert _run(_shape(), 2, _layer(q=17)) == 2                            # misaligned element


def test_what_the_tensor_cores_do_not_cover_is_unsupported():
    assert _run(_shape(dt=F32, D=64), 2, _layer(ks=64)) == 2               # fp32: no kind::f16 operands
    for D in (32, 96, 256):                                                # row widths outside {64, 80, 128}
        assert _run(_shape(D=D), 2, _layer(ks=D)) == 2, D
        assert _ws(_shape(D=D), 2, _layer(ks=D)) == -1, D
    for D in (64, 80, 128):
        assert _ws(_shape(D=D), 2, _layer(ks=D)) > 0, D
        assert _ws(_shape(D=D, dt=F16), 2, _layer(ks=D)) > 0, D
    assert _run(_shape(H=1), 129, _layer()) == 2                           # more than 128 query heads per KV head
    assert _run(_shape(), 2, _layer(q=1032)) == 2                          # q base 8-byte aligned: no tensor map
    assert _run(_shape(), 2, _layer(qs=(8192, 1028, 128))) == 2            # q head stride of 2056 bytes
    assert _run(_shape(), 2, _layer(qs=(8196, 1024, 128))) == 2            # q batch stride
    assert _run(_shape(), 2, _layer(qs=(8192, 1024, 132))) == 2            # q position stride
    assert _ws(_shape(), 2, _layer(qs=(8192, 1024, 132))) == -1


def test_a_mask_allows_more_queries_than_keys_and_nothing_to_do_is_ok():
    s = _shape()
    assert _ws(s, 2, _layer(mask=16, n_query=120, key_len=100)) > 0
    assert _lib().kvc_h2o_accumulate_qk_tc(s, 2, 0, None, 0.9, None, 0, None) == 0
    rec = _layer(key_len=0, n_query=1, lo=0, hi=0, mask=16)
    assert _ws(s, 2, rec) == 0
    assert _run(s, 2, rec, ws=0, ws_bytes=0) == 0


@pytest.mark.parametrize("G,T,tiles", [(1, 1, 1), (1, 128, 1), (1, 129, 2), (4, 32, 1), (4, 33, 2), (4, 4096, 128),
                                       (8, 1, 1), (8, 17, 2), (3, 42, 1), (3, 43, 2), (128, 5, 5)])
@pytest.mark.parametrize("B,H", [(1, 8), (3, 2)])
def test_workspace_arithmetic(G, T, tiles, B, H):
    """One fp32 lse2 per row of every 128-row query tile (G heads x 128 // G positions), per (b, KV head); 256-byte
    aligned per layer; a layer with no keys needs nothing."""
    assert -(-T // (128 // G)) == tiles
    one = -(-(B * H * tiles * 128 * 4) // 256) * 256
    s = _shape(B=B, H=H)
    rec = _layer(key_len=max(T, 100), n_query=T, lo=0, hi=0)
    assert _ws(s, G, rec) == one
    assert _ws(s, G, rec * 3, n=3) == 3 * one
    assert _ws(s, G, rec + _layer(key_len=0, n_query=1, lo=0, hi=0, mask=16), n=2) == one
    assert _ws(s, 0, rec) == -1


def _slab(**kw):
    return H2OScoreSlab(start_size=4, heavy_hitter_size=16, recent_size=40, num_layers=2, num_heads=8,
                        tensor_cores=True, **kw)


def test_manager_refusals_name_the_reason(monkeypatch):
    """fp32 and head dims outside {64, 80, 128} raise ValueError naming the reason, before anything is allocated or
    launched.  Meta tensors stand in for CUDA ones: the refusal comes before any device work."""
    monkeypatch.setattr(_engine, "_require_cuda", lambda t, what: None)
    m = _slab()
    assert m.tensor_cores and not H2OScoreSlab().tensor_cores
    for dt, D, reason in [(torch.float32, 128, "float32"), (torch.bfloat16, 96, "head_dim 96"),
                          (torch.float16, 32, "head_dim 32"), (torch.bfloat16, 256, "head_dim 256")]:
        q = torch.empty(1, 8, 4, D, dtype=dt, device="meta")
        k = torch.empty(1, 2, 16, D, dtype=dt, device="meta")
        with pytest.raises(ValueError, match=reason):
            m.update_from_queries([q], [k])
    assert m._acc is None
