"""Beam search on the slab cache (kvc_batch_reorder): the in-place batch gather of K, V, key norms and the per-row
score state against torch's index_select, one launch, no synchronisation, CUDA-graph replay, transformers' beam search
on slab.as_hf_cache(), and beam search with compression in lockstep with the function path."""

import pytest
import torch

import kvcompress
from kvcompress import H2OScoreSlab, KVSlabCache, SnapKVQueryWindow, _engine
from kvcompress.evaluate import new_slab_for_model

pytestmark = pytest.mark.gpu

BITS = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}


def indices(B):
    g = torch.Generator().manual_seed(B)
    out = {
        "identity": list(range(B)),
        "permutation": torch.randperm(B, generator=g).tolist(),
        "cycle": [(b + 1) % B for b in range(B)],
        "duplicates": [b // 2 for b in range(B)],
        "fork": [0] * B,
        "reversed": list(range(B))[::-1],
    }
    return out


def full_view(t, pitch):
    """t with its padding rows past capacity (the slab's pitch) visible."""
    shape = list(t.shape)
    shape[3] = pitch
    return t.as_strided(shape, t.stride())


def fill_random(slab, seed):
    g = torch.Generator(device=slab.device).manual_seed(seed)
    for t in (full_view(slab.k, slab.pitch), full_view(slab.v, slab.pitch), slab.n):
        bits = t.view(BITS[slab.dtype])
        bits.copy_(torch.randint(-2 ** 15, 2 ** 15, bits.shape, generator=g, device=slab.device, dtype=torch.int32))


def expected(slab, before, idx):
    """Every byte of K, V (padding included) and the norms after index_select of each layer's valid rows."""
    want = [t.clone() for t in before]
    for l, n in enumerate(slab.lengths):
        for w, b in zip(want, before):
            w[l, :, :, :n] = b[l].index_select(0, idx)[:, :, :n]
    return want


def state(slab):
    return [full_view(slab.k, slab.pitch).clone(), full_view(slab.v, slab.pitch).clone(), slab.n.clone()]


def same_bits(a, b):
    return torch.equal(a.view(BITS[a.dtype]), b.view(BITS[b.dtype]))


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("row_bytes", [16, 160, 256, 512, 2048])
@pytest.mark.parametrize("B", [1, 3, 8, 64])
def test_slab_reorder_matches_index_select(B, row_bytes, dtype):
    e = torch.empty((), dtype=dtype).element_size()
    # 256- and 512-byte rows at capacity 64 get pitch padding past the capacity (the bytes must stay untouched); the
    # other widths use an odd capacity, where the norm rows are only 2- or 4-byte aligned
    cap = 64 if row_bytes in (256, 512) else 41
    slab = KVSlabCache(4, B, 2, row_bytes // e, cap, dtype)
    assert (slab.pitch > cap) == (cap == 64)
    slab.lengths = [0, 17, cap, 1]
    cases = dict(indices(B))
    cases["out of range (clamped)"] = [B + 7 if b % 2 else -3 for b in range(B)]
    for name, idx in cases.items():
        for itype in (torch.int32, torch.int64):
            fill_random(slab, hash((name, itype == torch.int64)) % 1000)
            before = state(slab)
            dev_idx = torch.tensor(idx, dtype=itype, device="cuda")
            slab.reorder_(dev_idx)
            clamped = dev_idx.clamp(0, B - 1).long()
            for got, want in zip(state(slab), expected(slab, before, clamped)):
                assert same_bits(got, want), (name, itype)
            assert slab.lengths == [0, 17, cap, 1]


def tiny_followers(B, carry):
    """An H2OScoreSlab (GQA: 8 query heads over 2 KV heads) with accumulators of different lengths per layer, and a
    SnapKVQueryWindow with one layer partly filled and one full."""
    L, Hq, Hkv, D, W = 2, 8, 2, 64, 8
    g = torch.Generator(device="cuda").manual_seed(5)
    h2o = H2OScoreSlab(start_size=2, heavy_hitter_size=4, recent_size=4, num_layers=L, num_heads=Hq,
                       carry_scores=carry)
    keys = [torch.randn(B, Hkv, n, D, generator=g, device="cuda").bfloat16() for n in (10, 23)]
    for _ in range(2):
        q = [torch.randn(B, Hq, 1, D, generator=g, device="cuda").bfloat16() for _ in range(L)]
        h2o.update_from_queries(q, keys)
    win = SnapKVQueryWindow(L, B, Hq, D, W, torch.bfloat16)
    win.push([torch.randn(B, Hq, 5, D, generator=g, device="cuda").bfloat16(),
              torch.randn(B, Hq, 11, D, generator=g, device="cuda").bfloat16()])
    return h2o, win


@pytest.mark.parametrize("carry", [False, True])
def test_followers_move_with_the_slab_in_one_launch(carry):
    B = 4
    h2o, win = tiny_followers(B, carry)
    slab = KVSlabCache(2, B, 2, 64, 32, torch.bfloat16)
    slab.lengths = [9, 32]
    fill_random(slab, 1)
    before = state(slab)
    acc0 = {l: h2o.accumulated_attention[l].clone() for l in (0, 1)}
    win0 = [q.clone() for q in win.queries]
    idx = torch.tensor([2, 2, 0, 3], device="cuda")
    n0 = _engine.launch_count()
    slab.reorder_(idx, h2o, win)
    assert _engine.launch_count() - n0 == 1
    for got, want in zip(state(slab), expected(slab, before, idx)):
        assert same_bits(got, want)
    for l in (0, 1):
        assert torch.equal(h2o.accumulated_attention[l], acc0[l].index_select(0, idx))
        n = win.filled[l]
        assert torch.equal(win.queries[l][:, :, :n], win0[l][:, :, :n].index_select(0, idx))
        assert same_bits(win.queries[l][:, :, n:], win0[l][:, :, n:])     # rows past `filled` are not touched
    assert h2o._scored == {}
    # the function path: each follower on its own
    idx2 = torch.tensor([1, 0, 3, 3], device="cuda", dtype=torch.int32)
    acc1 = {l: h2o.accumulated_attention[l].clone() for l in (0, 1)}
    win1 = [q.clone() for q in win.queries]
    n0 = _engine.launch_count()
    h2o.reorder_(idx2)
    win.reorder_(idx2.cpu())
    assert _engine.launch_count() - n0 == 2
    for l in (0, 1):
        assert torch.equal(h2o.accumulated_attention[l], acc1[l].index_select(0, idx2.long()))
        assert torch.equal(win.queries[l][:, :, :win.filled[l]],
                           win1[l][:, :, :win.filled[l]].index_select(0, idx2.long()))
    # a window of another shape replaces the first one (possibly at the same address): the reorder follows the new one
    del win, win0, win1
    small = SnapKVQueryWindow(2, B, 8, 64, 4, torch.bfloat16)
    small.push([torch.randn(B, 8, 3, 64, device="cuda").bfloat16(), torch.randn(B, 8, 6, 64, device="cuda").bfloat16()])
    small_before = [q.clone() for q in small.queries]
    slab.reorder_(idx, small)
    for l in (0, 1):
        n = small.filled[l]
        assert torch.equal(small.queries[l][:, :, :n], small_before[l][:, :, :n].index_select(0, idx))
    empty = H2OScoreSlab(num_layers=2)
    n0 = _engine.launch_count()
    empty.reorder_(idx)
    slab.reorder_(idx, empty)
    assert _engine.launch_count() - n0 == 1                         # a manager with no buffers moves nothing


def test_no_sync_and_graph_replay():
    B = 8
    slab = KVSlabCache(3, B, 4, 80, 64, torch.bfloat16)
    slab.lengths = [64, 30, 5]
    _, win = tiny_followers(B, True)
    fill_random(slab, 2)
    idx = torch.tensor([3, 3, 7, 0, 1, 1, 6, 2], device="cuda")
    slab.reorder_(idx, win)                                          # packs the records (host work, outside the mode)
    torch.cuda.synchronize()
    start = state(slab) + [q.clone() for q in win.queries]
    torch.cuda.set_sync_debug_mode("error")
    try:
        slab.reorder_(idx, win)
        slab.reorder_(idx, win)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    eager = state(slab) + [q.clone() for q in win.queries]
    graph = torch.cuda.CUDAGraph()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph):
            slab.reorder_(idx, win)
    torch.cuda.current_stream().wait_stream(stream)
    # capture records without running: restore the starting bytes, then replay the captured call twice
    for t, s in zip([full_view(slab.k, slab.pitch), full_view(slab.v, slab.pitch), slab.n] + win.queries, start):
        t.copy_(s)
    graph.replay()
    graph.replay()
    torch.cuda.synchronize()
    for got, want in zip(state(slab) + win.queries, eager):
        assert same_bits(got, want)


def tiny_llama_gqa(dtype=torch.float32):
    from transformers import LlamaConfig, LlamaForCausalLM

    torch.manual_seed(0)
    cfg = LlamaConfig(vocab_size=256, hidden_size=512, num_hidden_layers=3, num_attention_heads=8,
                      num_key_value_heads=2, intermediate_size=256, max_position_embeddings=512)
    return LlamaForCausalLM(cfg).eval().cuda().to(dtype)


@pytest.mark.parametrize("kind", ["neox", "llama_gqa"])
def test_hf_beam_search_on_the_slab_matches_dynamic_cache(kind):
    """Fails without a reorder: each beam would keep attending to the cache of the sequence it started in."""
    from transformers import DynamicCache

    if kind == "neox":
        from golden.harness_cases import tiny_model_and_ids

        model, ids = tiny_model_and_ids("cuda")
        ids = ids[:, :24].cuda()
    else:
        model = tiny_llama_gqa()
        ids = torch.randint(0, 256, (1, 24), generator=torch.Generator().manual_seed(1)).cuda()
    kw = dict(num_beams=4, num_return_sequences=4, max_new_tokens=16, min_new_tokens=16, do_sample=False,
              return_dict_in_generate=True, output_scores=True, pad_token_id=0)
    with torch.inference_mode():
        ref = model.generate(ids, past_key_values=DynamicCache(), **kw)
        slab = new_slab_for_model(model, 4, capacity=64)
        got = model.generate(ids, past_key_values=slab.as_hf_cache(), **kw)
    assert torch.equal(got.sequences, ref.sequences)
    assert torch.allclose(got.sequences_scores, ref.sequences_scores, atol=1e-5, rtol=0)


# ------------------------------------------------------------------ beam search with compression, lockstep
METHODS = {
    "h2o_l2": dict(start_size=4, heavy_hitter_size=8, recent_size=12),
    "streaming_llm": dict(start_size=4, recent_size=20),
    "snapkv_lite": dict(observation_window=8, keep_size=24, pooling_kernel=5),
    "snapkv_lite_queries": dict(observation_window=8, keep_size=24, pooling_kernel=5),
    "h2o_attention": dict(start_size=4, heavy_hitter_size=8, recent_size=12),
}


@pytest.mark.parametrize("method", list(METHODS))
def test_beam_search_with_compression_lockstep(method):
    """A manual beam loop (log-softmax, top-k over beams x vocab, beam_idx) drives two caches from the same forward:
    the slab (compress_ + reorder_, followers moved in the same launch) and lists of tensors (the compress function +
    index_select, followers reordered in torch).  The new rows of every forward go to both; after every compression and
    every reorder the two caches and follower states are bit-identical, and so are the tokens they lead to."""
    kw = dict(METHODS[method], skip_layers=[])
    model = tiny_llama_gqa(torch.bfloat16)
    L, V, nb = model.config.num_hidden_layers, model.config.vocab_size, 4
    slab = new_slab_for_model(model, nb, capacity=64)
    cache = slab.as_hf_cache()
    win_a = win_b = h2o_a = h2o_b = None
    fn_name = "snapkv_lite" if method == "snapkv_lite_queries" else method
    fn = kvcompress.get_compress_fn(fn_name)
    if method == "snapkv_lite_queries":
        win_a, win_b = (SnapKVQueryWindow.for_model(model, nb, 8) for _ in range(2))
    if method == "h2o_attention":
        h2o_a, h2o_b = (H2OScoreSlab(4, 8, 12, num_layers=L, num_heads=model.config.num_attention_heads,
                                     carry_scores=True) for _ in range(2))
    prompt = torch.randint(0, V, (1, 20), generator=torch.Generator().manual_seed(2)).cuda().expand(nb, -1)
    kv_b = None
    beam_scores = torch.tensor([0.0] + [float("-inf")] * (nb - 1), device="cuda")
    step_in = prompt
    with torch.inference_mode():
        for step in range(14):
            with kvcompress.capture_queries(model) as cap:
                out = model(step_in, past_key_values=cache, use_cache=True)
            T = step_in.size(1)
            new = [(k[:, :, -T:].clone(), v[:, :, -T:].clone()) for k, v in slab]
            kv_b = new if kv_b is None else [(torch.cat([k, nk], 2), torch.cat([v, nv], 2))
                                             for (k, v), (nk, nv) in zip(kv_b, new)]
            if win_a is not None:
                win_a.push(cap)
                win_b.push(cap)
            if h2o_a is not None:
                h2o_b.update_from_queries(cap.queries, [k for k, _ in kv_b], cap.masks, cap.scaling)
                slab.compress_(method, h2o_manager=h2o_a, attention_queries=cap, **kw)
                kv_b = fn(kv_b, h2o_manager=h2o_b, **kw)
            elif win_a is not None:
                if slab.lengths[0] > kw["keep_size"]:
                    slab.compress_(fn_name, obs_queries=win_a, **kw)
                    kv_b = fn(kv_b, obs_queries=win_b, **kw)
            else:
                slab.compress_(method, **kw)
                kv_b = fn(kv_b, **kw)
            for l in range(L):
                assert torch.equal(slab[l][0], kv_b[l][0]) and torch.equal(slab[l][1], kv_b[l][1]), (step, l)
            logp = torch.log_softmax(out.logits[:, -1].float(), dim=-1)
            top = (beam_scores[:, None] + logp).view(-1).topk(nb)
            beam_idx, tokens, beam_scores = top.indices // V, top.indices % V, top.values
            slab.reorder_(beam_idx, *[f for f in (win_a, h2o_a) if f is not None])
            kv_b = [(k.index_select(0, beam_idx), v.index_select(0, beam_idx)) for k, v in kv_b]
            if win_b is not None:
                win_b._buf.copy_(win_b._buf.index_select(1, beam_idx))
            if h2o_b is not None:
                h2o_b._acc.copy_(h2o_b._acc.index_select(1, beam_idx))
                h2o_b._scored = {}
            for l in range(L):
                assert torch.equal(slab[l][0], kv_b[l][0]) and torch.equal(slab[l][1], kv_b[l][1]), (step, l)
            step_in = tokens[:, None]
    assert slab.lengths[0] <= 24 + 1
    for l in range(L):
        if win_a is not None:
            assert win_a.filled == win_b.filled and torch.equal(win_a.queries[l], win_b.queries[l])
        if h2o_a is not None:
            assert h2o_a._lens == h2o_b._lens
            assert torch.equal(h2o_a.accumulated_attention[l], h2o_b.accumulated_attention[l])


def test_integration_recipe_generate_with_compression():
    """INTEGRATION.md's recipe: model.generate with beam search, a LogitsProcessor that pushes the captured queries
    into the window and compresses the slab, and a cache whose reorder moves the window with the beams."""
    from transformers import LogitsProcessor, LogitsProcessorList

    model = tiny_llama_gqa(torch.bfloat16)
    W, keep, beams = 8, 24, 4
    slab = new_slab_for_model(model, beams, capacity=64)
    window = SnapKVQueryWindow.for_model(model, beams, W)

    class CompressEachStep(LogitsProcessor):
        def __init__(self, cap):
            self.cap = cap

        def __call__(self, input_ids, scores):
            window.push(self.cap)
            if slab.lengths[0] > keep:
                slab.compress_("snapkv_lite", observation_window=W, keep_size=keep, skip_layers=[], obs_queries=window)
            return scores

    ids = torch.randint(0, 256, (1, 20), generator=torch.Generator().manual_seed(4)).cuda()
    with torch.inference_mode(), kvcompress.capture_queries(model) as cap:
        out = model.generate(ids, past_key_values=slab.as_hf_cache(followers=[window]), num_beams=beams,
                             max_new_tokens=20, min_new_tokens=20, do_sample=False, pad_token_id=0,
                             logits_processor=LogitsProcessorList([CompressEachStep(cap)]))
    assert out.shape == (1, 40)
    assert slab.lengths == [keep] * model.config.num_hidden_layers
