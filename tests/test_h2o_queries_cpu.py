"""H2O scores from queries without a GPU: the C ABI of kvc_h2o_accumulate_qk (struct layout, argument checks that run
before any CUDA call, workspace arithmetic) and kvcompress.capture_queries on tiny transformers models on the CPU."""

import ctypes
import math

import pytest
import torch

import kvcompress
from kvcompress import _engine

BF16, F32 = 2, 0


def _shape(B=1, H=2, D=64, dt=BF16):
    return _engine._SHAPE.pack(B, H, D, dt, 0)


def _layer(q=16, k=16, mask=0, acc=16, score=16, n_query=1, key_len=100, prev_len=-1, lo=4, hi=50, ks=64, scaling=0.125):
    return _engine._H2O_QK.pack(q, 1000, 100, 64, k, ks * 200, ks * 100, ks, mask, 1000, 100, acc, 800, 200, score,
                                scaling, n_query, key_len, prev_len, lo, hi)


def _lib():
    return _engine.load_library()


def _ws(shape, group, recs, n=1):
    return _lib().kvc_h2o_qk_workspace_bytes(shape, group, n, recs)


def _run(shape, group, recs, n=1, ws=1 << 20, ws_bytes=1 << 20):
    return _lib().kvc_h2o_accumulate_qk(shape, group, n, recs, 0.9, ctypes.c_void_p(ws), ws_bytes, None)


def test_struct_matches_the_header():
    assert _engine._H2O_QK.size == 144


def test_invalid_arguments_are_refused_before_any_cuda_call():
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
    assert _run(s, 0, None, n=0) == 1                                      # group < 1 with nothing to do


def test_unsupported_shapes_are_refused_before_any_cuda_call():
    assert _run(_shape(dt=7), 2, _layer()) == 2                            # dtype
    assert _run(_shape(D=60), 2, _layer()) == 2                            # 120-byte rows: not a multiple of 16
    assert _run(_shape(D=264), 2, _layer()) == 2                           # 528-byte rows: above 512
    assert _run(_shape(D=256), 2, _layer(ks=256)) != 2                     # 512-byte bf16 rows are covered
    assert _run(_shape(D=136, dt=F32), 2, _layer(ks=136)) == 2             # 544-byte fp32 rows
    assert _run(_shape(D=68), 2, _layer(ks=68)) == 2                       # 136-byte rows: D * e = 136, not 16-aligned
    assert _run(_shape(), 2, _layer(k=24)) == 2                            # K not 16-byte aligned
    assert _run(_shape(), 2, _layer(ks=60)) == 2                           # K row stride not 16-byte aligned
    assert _run(_shape(), 2, _layer(q=17)) == 2                            # misaligned element


def test_a_mask_allows_more_queries_than_keys_and_nothing_to_do_is_ok():
    s = _shape()
    rec = _layer(mask=16, n_query=120, key_len=100)
    assert _ws(s, 2, rec) > 0
    assert _lib().kvc_h2o_accumulate_qk(s, 2, 0, None, 0.9, None, 0, None) == 0
    assert _ws(s, 2, _layer(key_len=0, n_query=1, lo=0, hi=0, mask=16)) == 0
    assert _run(s, 2, _layer(key_len=0, n_query=1, lo=0, hi=0, mask=16), ws=0, ws_bytes=0) == 0


@pytest.mark.parametrize("key_len,splits", [(1, 1), (128, 1), (129, 2), (513, 5), (4096, 32), (4097, 17),
                                            (32768, 32), (100000, 32)])
@pytest.mark.parametrize("B,H,G,T", [(1, 8, 4, 1), (2, 3, 1, 7)])
def test_workspace_arithmetic(key_len, splits, B, H, G, T):
    """(max, sum exp) as two fp32 per (b, KV head, query head of the group, query, key split), 256-byte aligned per
    layer; splits: at most 32 of a whole number of 128-row tiles each."""
    tiles = -(-key_len // 128)
    per = -(-tiles // min(32, tiles))
    assert -(-tiles // per) == splits
    one = B * H * G * T * splits * 8
    one = -(-one // 256) * 256
    s = _shape(B=B, H=H)
    rec = _layer(key_len=key_len, n_query=T, lo=0, hi=0, mask=16)
    assert _ws(s, G, rec) == one
    assert _ws(s, G, rec * 3, n=3) == 3 * one
    assert _ws(s, 0, rec) == -1


# ------------------------------------------------------------------ capture_queries on tiny models
def _neox():
    from transformers import GPTNeoXConfig, GPTNeoXForCausalLM

    torch.manual_seed(0)
    cfg = GPTNeoXConfig(vocab_size=128, hidden_size=256, num_hidden_layers=2, num_attention_heads=4,
                        intermediate_size=256, max_position_embeddings=256, rotary_pct=0.25)
    return GPTNeoXForCausalLM(cfg).eval()


def _llama_gqa():
    from transformers import LlamaConfig, LlamaForCausalLM

    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=128, hidden_size=256, num_hidden_layers=2, num_attention_heads=8,
                      num_key_value_heads=2, intermediate_size=256, max_position_embeddings=256)
    return LlamaForCausalLM(cfg).eval()


MODELS = {"neox": _neox, "llama_gqa": _llama_gqa}


def _probs_from_records(cap, layer):
    """§ the contract: fp32 logits scaling * q . k over the un-repeated keys, visible = mask or the causal rule."""
    q, k, mask, scaling = cap.queries[layer], cap.keys[layer], cap.masks[layer], cap.scaling[layer]
    B, Hq, T, D = q.shape
    S = k.size(2)
    kr = k.repeat_interleave(Hq // k.size(1), dim=1)
    s = scaling * torch.matmul(q.double(), kr.double().transpose(-1, -2))
    if mask is None:
        vis = torch.arange(S).view(1, S) <= (S - T + torch.arange(T)).view(T, 1)
        vis = vis.view(1, 1, T, S)
    else:
        vis = mask[..., :S]
    s = s.masked_fill(~vis, float("-inf"))
    p = torch.softmax(s, dim=-1).nan_to_num(0.0)
    return p.float(), vis


def _run_both(model, steps, attention_mask=None):
    """Run the same forwards under the capture and under eager + output_attentions; yield per step
    (capture, eager attentions, logits under the capture, logits under sdpa)."""
    from transformers import DynamicCache

    caches = {"cap": DynamicCache(), "eager": DynamicCache(), "sdpa": DynamicCache()}
    out = []
    pos = 0
    for ids in steps:
        T = ids.size(1)
        am = None if attention_mask is None else attention_mask[:, :pos + T]
        with torch.inference_mode():
            with kvcompress.capture_queries(model) as cap:
                got = model(ids, past_key_values=caches["cap"], use_cache=True, attention_mask=am)
            model.set_attn_implementation("sdpa")
            ref = model(ids, past_key_values=caches["sdpa"], use_cache=True, attention_mask=am)
            model.set_attn_implementation("eager")
            eager = model(ids, past_key_values=caches["eager"], use_cache=True, attention_mask=am,
                          output_attentions=True)
        out.append((cap, eager.attentions, got.logits, ref.logits))
        pos += T
    return out


@pytest.mark.parametrize("name", sorted(MODELS))
def test_capture_records_queries_keys_masks(name):
    """Plain prefill, a chunked prefill (materialised mask) and decode: outputs equal SDPA bit for bit, keys are the
    un-repeated [B, Hkv, S, D], and the softmax rebuilt from the records equals eager attention within 1e-6."""
    model = _neox() if name == "neox" else _llama_gqa()
    model.set_attn_implementation("sdpa")
    cfg = model.config
    Hq = cfg.num_attention_heads
    Hkv = getattr(cfg, "num_key_value_heads", None) or Hq
    D = cfg.hidden_size // Hq
    ids = torch.randint(0, cfg.vocab_size, (1, 33), generator=torch.Generator().manual_seed(3))
    steps = [ids[:, :24], ids[:, 24:32], ids[:, 32:33]]
    for (cap, attentions, got, ref), T, S in zip(_run_both(model, steps), (24, 8, 1), (24, 32, 33)):
        assert torch.equal(got, ref)
        for layer in range(cfg.num_hidden_layers):
            assert cap.queries[layer].shape == (1, Hq, T, D)
            assert cap.keys[layer].shape == (1, Hkv, S, D)
            assert cap.scaling[layer] == pytest.approx(D ** -0.5)
            p, _ = _probs_from_records(cap, layer)
            assert p.shape == attentions[layer].shape
            assert torch.allclose(p, attentions[layer].float(), atol=1e-6, rtol=0), (T, layer)
    assert model.config._attn_implementation == "eager"  # what _run_both left


def test_capture_left_padded_batch():
    """A left-padded batch of 2: the rebuilt softmax of every real query row equals eager attention."""
    model = _llama_gqa()
    cfg = model.config
    ids = torch.randint(0, cfg.vocab_size, (2, 10), generator=torch.Generator().manual_seed(4))
    am = torch.ones(2, 10, dtype=torch.long)
    am[0, :3] = 0
    (cap, attentions, got, ref), = _run_both(model, [ids], attention_mask=am)
    assert torch.equal(got, ref)
    for layer in range(cfg.num_hidden_layers):
        assert cap.masks[layer] is not None and cap.masks[layer].dtype == torch.bool
        assert tuple(cap.masks[layer].shape) == (2, 1, 10, 10)
        p, _ = _probs_from_records(cap, layer)
        real = am.bool().view(2, 1, 10, 1).expand_as(p)   # padded query rows are not compared
        assert torch.allclose(p[real], attentions[layer].float()[real], atol=1e-6, rtol=0)


def test_capture_restores_the_implementation_even_after_an_exception():
    model = _neox()
    model.set_attn_implementation("eager")
    with kvcompress.capture_queries(model) as cap:
        assert model.config._attn_implementation == "kvcompress_sdpa"
        assert isinstance(cap, kvcompress.QueryCapture)
    assert model.config._attn_implementation == "eager"
    with pytest.raises(RuntimeError, match="boom"):
        with kvcompress.capture_queries(model):
            raise RuntimeError("boom")
    assert model.config._attn_implementation == "eager"


def test_capture_refuses_what_it_cannot_reproduce():
    from transformers import AttentionInterface

    from kvcompress.capture import ATTN_NAME

    model = _neox()
    with kvcompress.capture_queries(model):
        fn = AttentionInterface()[ATTN_NAME]
        attn = model.gpt_neox.layers[0].attention
        q = torch.randn(1, 4, 3, 64)
        for kw in (dict(softcap=30.0), dict(s_aux=torch.zeros(4)), dict(sinks=torch.zeros(4)), dict(dropout=0.1)):
            with pytest.raises(ValueError):
                fn(attn, q, q, q, None, **kw)


def test_h2o_attention_manager_has_no_query_path():
    m = kvcompress.H2OAttentionManager(num_layers=1, num_heads=2)
    cap = kvcompress.QueryCapture(1)
    kv = [(torch.zeros(1, 2, 8, 16), torch.zeros(1, 2, 8, 16))]
    with pytest.raises(ValueError, match="H2OScoreSlab"):
        kvcompress.h2o_attention_compress(kv, h2o_manager=m, attention_queries=cap, start_size=1,
                                          heavy_hitter_size=2, recent_size=2)
    with pytest.raises(ValueError, match="H2OScoreSlab"):
        kvcompress.h2o_attention_compress(kv, attention_queries=cap, start_size=1, heavy_hitter_size=2, recent_size=2)


def test_update_from_queries_refuses_a_per_head_mask():
    m = kvcompress.H2OScoreSlab(num_layers=1, num_heads=4)
    q, k = torch.zeros(1, 4, 2, 16), torch.zeros(1, 2, 8, 16)
    with pytest.raises(ValueError, match="per-head"):
        m.update_from_queries([q], [k], masks=[torch.ones(1, 4, 2, 8, dtype=torch.bool)])


def test_exports():
    assert "capture_queries" in kvcompress.__all__ and "QueryCapture" in kvcompress.__all__
    assert math.isclose(kvcompress.QueryCapture(2).num_layers, 2)
