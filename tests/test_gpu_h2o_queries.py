"""-m gpu: H2OScoreSlab.update_from_queries — the H2O attention mass rebuilt on the device from the queries and the
cached keys (kvc_h2o_accumulate_qk) — against fp64 torch logits -> softmax -> .to(dtype) -> the torch manager's update,
and the capture path (kvcompress.capture_queries, SDPA) against the eager output_attentions path."""

import json
import os

import pytest
import torch

import kvcompress
from kvcompress import H2OAttentionManager, H2OScoreSlab, KVSlabCache, QueryCapture, _engine

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
MANTISSA = {torch.bfloat16: 7, torch.float16: 10}
KW = dict(start_size=4, heavy_hitter_size=16, recent_size=40)


def assert_close_ulp(got, want, what, rtol=1e-5):
    """fp32: 1e-5 relative — the logits are fp32 dot products of D terms (relative error ~D * 2^-24 of the sum of
    |terms|), exp and the max-shifted log-sum-exp add a few ulps, and the query and head sums add T and Hq terms; 1e-5
    covers that with a margin for D <= 128.
    16-bit: within one unit in the last place of the larger magnitude, except at rounding near-ties: a probability
    whose fp32 value lies within ~1e-6 of a rounding boundary of the dtype can round the other way than the fp64
    reference's, which moves the mass by one ulp of that probability, and the update's own rounding of
    round(acc * decay) + mass can then land one more ulp away.  So at most 2 ulps anywhere, and beyond 1 ulp on at most
    0.1% of the entries."""
    g, w = got.double(), want.double()
    if got.dtype == torch.float32:
        bound = rtol * torch.maximum(g.abs(), w.abs()) + 1e-30
        bad = (g - w).abs() > bound
        assert not bool(bad.any()), f"{what}: {int(bad.sum())} entries off, worst {float((g - w).abs().max())}"
        return
    mag = torch.maximum(g.abs(), w.abs()).clamp_min(2.0 ** -14 if got.dtype == torch.float16 else 2.0 ** -126)
    ulp = torch.exp2(torch.floor(torch.log2(mag)) - MANTISSA[got.dtype])
    diff = (g - w).abs()
    assert not bool((diff > 2 * ulp).any()), f"{what}: {int((diff > 2 * ulp).sum())} entries beyond 2 ulps"
    n1 = int((diff > ulp).sum())
    assert n1 <= max(1, diff.numel() // 1000), f"{what}: {n1} of {diff.numel()} entries beyond 1 ulp"


def ref_probs(q, k, mask=None, scaling=None):
    """The contract in fp64: logits, visibility (mask or causal), softmax, 0 where invisible, then .to(dtype)."""
    B, Hq, T, D = q.shape
    S = k.size(2)
    scaling = D ** -0.5 if scaling is None else scaling
    kr = k.double().repeat_interleave(Hq // k.size(1), dim=1)
    s = scaling * torch.matmul(q.double(), kr.transpose(-1, -2))
    if mask is None:
        vis = (torch.arange(S, device=q.device).view(1, S) <=
               (S - T + torch.arange(T, device=q.device)).view(T, 1)).view(1, 1, T, S)
    else:
        vis = (mask[:, 0] if mask.dim() == 4 else mask)[..., :S].unsqueeze(1)
    p = torch.softmax(s.masked_fill(~vis, float("-inf")), dim=-1).nan_to_num(0.0)
    return p.masked_fill(~vis, 0.0).to(q.dtype)


def inputs(B, Hkv, G, T, K, D, dtype, gen, cap_extra=24, scale=1.0):
    """Queries and keys; the keys are a strided view [B, Hkv, K, D] of a longer slab-like buffer."""
    q = (scale * torch.randn(B, Hkv * G, T, D, generator=gen, device="cuda")).to(dtype)
    kbuf = torch.randn(B, Hkv, K + cap_extra, D, generator=gen, device="cuda").to(dtype)
    return q, kbuf[:, :, :K]


def pair(L, Hq, capacity=None):
    args = dict(KW, num_layers=L, num_heads=Hq, decay_factor=0.9)
    return H2OAttentionManager(**args), H2OScoreSlab(capacity=capacity, **args)


def check_step(ref, dev, L, B, K, what):
    for l in range(L):
        acc = dev.accumulated_attention[l]
        assert_close_ulp(acc, ref.accumulated_attention[l], f"{what} acc layer {l}")
        lo, hi = KW["start_size"], K - KW["recent_size"]
        if hi > lo:
            assert_close_ulp(dev._score_row(l, B, hi - lo), acc[:, :, lo:hi].sum(dim=1), f"{what} score layer {l}")


@pytest.mark.parametrize("dtype", ["f32", "bf16", "f16"])
@pytest.mark.parametrize("G,T,K,D", [(1, 1, 301, 64), (4, 1, 1000, 128), (4, 7, 300, 128), (8, 128, 333, 80),
                                     (4, 264, 264, 96), (8, 1, 517, 64)])
def test_accumulators_and_score_rows_match_the_reference(dtype, G, T, K, D):
    """One step at a time from the device's state: the accumulators within 1 ulp (16-bit) / 1e-5 (fp32) of fp64
    logits -> softmax -> .to(dtype) -> the torch manager's update, the score row with the head sum."""
    dt = DT[dtype]
    L, B, Hkv = 2, 2, 2
    ref, dev = pair(L, Hkv * G)
    gen = torch.Generator(device="cuda").manual_seed(G * 1000 + T + K)
    for step in range(2):
        Ks = K + step * min(T, 5)   # the second step grows the cache (and decays the first step's mass)
        Ts = min(T, Ks)
        qk = [inputs(B, Hkv, G, Ts, Ks, D, dt, gen, scale=2.0) for _ in range(L)]
        if step:
            ref.accumulated_attention = {l: dev.accumulated_attention[l].clone() for l in range(L)}
        ref.update_attention_scores([ref_probs(q, k) for q, k in qk])
        dev.update_from_queries([q for q, _ in qk], [k for _, k in qk])
        assert dev.current_seq_len == Ks
        check_step(ref, dev, L, B, Ks, f"step {step}")


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_growing_repeated_shrinking_skipped_and_none_layers(dtype):
    """The state transitions of update_attention_scores: growth, a repeated key length (the harness's double update),
    a shrink (reset), skipped and None layers, buffer doubling from a small capacity."""
    dt = DT[dtype]
    L, B, Hkv, G, D = 4, 2, 2, 3, 64
    ref, dev = pair(L, Hkv * G, capacity=64)
    gen = torch.Generator(device="cuda").manual_seed(11)
    for step, (K, skip, none) in enumerate([(100, [], []), (101, [1], []), (101, [], [2]), (150, [], []),
                                            (150, [0], []), (90, [], []), (91, [3], [1]), (300, [], [])]):
        qk = [inputs(B, Hkv, G, 1, K, D, dt, gen) for _ in range(L)]
        queries = [None if l in none else q for l, (q, _) in enumerate(qk)]
        repeats = 2 if step == 2 else 1
        for _ in range(repeats):
            ref.accumulated_attention = {l: dev.accumulated_attention[l].clone() for l in dev.accumulated_attention}
            ref.current_seq_len = dev.current_seq_len
            ref.update_attention_scores([None if q is None else ref_probs(q, k) for q, (_, k) in zip(queries, qk)], skip)
            dev.update_from_queries(queries, [k for _, k in qk], skip_layers=skip)
            assert dev.current_seq_len == ref.current_seq_len
            assert sorted(dev.accumulated_attention) == sorted(ref.accumulated_attention)
            for l, want in ref.accumulated_attention.items():
                got = dev.accumulated_attention[l]
                assert got.shape == want.shape, (step, l)
                assert_close_ulp(got, want, f"step {step} layer {l}")
    assert dev.capacity >= 300


def test_masks():
    """Padded key columns get exactly 0; a fully masked query row adds nothing; a [B, 1, T, S] mask whose batch stride
    is 0 works."""
    L, B, Hkv, G, T, K, D = 1, 3, 2, 2, 5, 200, 64
    gen = torch.Generator(device="cuda").manual_seed(12)
    q, k = inputs(B, Hkv, G, T, K, D, torch.float32, gen)
    mask = torch.ones(B, 1, T, K, dtype=torch.bool, device="cuda")
    mask[0, :, :, :30] = False            # entry 0: 30 left-padded key columns
    mask[1, :, 2, :] = False              # entry 1: query 2 sees nothing
    mask[2] = torch.tril(torch.ones(T, K, dtype=torch.bool, device="cuda"), diagonal=K - T)
    ref, dev = pair(L, Hkv * G)
    ref.update_attention_scores([ref_probs(q, k, mask)])
    dev.update_from_queries([q], [k], masks=[mask])
    acc = dev.accumulated_attention[0]
    assert bool((acc[0, :, :30] == 0).all())
    check_step(ref, dev, L, B, K, "mask")
    # query 2 of entry 1 contributes nothing: the same as the other queries alone
    _, alone = pair(L, Hkv * G)
    keep = [0, 1, 3, 4]
    m2 = mask[1:2, :, keep]
    alone.update_from_queries([q[1:2, :, keep]], [k[1:2]], masks=[m2])
    assert torch.equal(alone.accumulated_attention[0][0], acc[1])
    # one [1, 1, T, S] mask for the batch: expanded with a zero batch stride
    causal = torch.tril(torch.ones(T, K, dtype=torch.bool, device="cuda"), diagonal=K - T).view(1, 1, T, K)
    _, a = pair(L, Hkv * G)
    _, b = pair(L, Hkv * G)
    a.update_from_queries([q], [k], masks=[causal.expand(B, 1, T, K)])
    b.update_from_queries([q], [k])
    assert torch.equal(a.accumulated_attention[0], b.accumulated_attention[0])


def test_determinism_and_independence_from_the_launch():
    """The same inputs give the same bits; a layer alone equals the same layer inside a multi-layer launch with other
    shapes; a batch entry alone equals the same entry inside a batch."""
    B, Hkv, G, D = 3, 2, 4, 128
    gen = torch.Generator(device="cuda").manual_seed(13)
    shapes = [(7, 900), (1, 4000), (33, 700)]
    qk = [inputs(B, Hkv, G, T, K, D, torch.bfloat16, gen, scale=2.0) for T, K in shapes]
    _, a = pair(3, Hkv * G)
    _, b = pair(3, Hkv * G)
    a.update_from_queries([q for q, _ in qk], [k for _, k in qk])
    b.update_from_queries([q for q, _ in qk], [k for _, k in qk])
    for l in range(3):
        assert torch.equal(a.accumulated_attention[l], b.accumulated_attention[l])
    for l in range(3):
        _, one = pair(3, Hkv * G)
        one.update_from_queries([q if i == l else None for i, (q, _) in enumerate(qk)], [k for _, k in qk])
        assert torch.equal(one.accumulated_attention[l], a.accumulated_attention[l]), l
        _, entry = pair(3, Hkv * G)
        entry.update_from_queries([q[1:2] if i == l else None for i, (q, _) in enumerate(qk)],
                                  [k[1:2] for _, k in qk])
        assert torch.equal(entry.accumulated_attention[l][0], a.accumulated_attention[l][1]), l


@pytest.mark.parametrize("T", [1, 256])
def test_long_keys(T):
    """B 1, Hq 32, Hkv 8, D 128, key_len 32768 (bf16) against the reference, two steps."""
    B, Hkv, G, K, D = 1, 8, 4, 32768, 128
    gen = torch.Generator(device="cuda").manual_seed(14 + T)
    ref, dev = pair(1, Hkv * G)
    for step in range(2):
        q, k = inputs(B, Hkv, G, T, K + step, D, torch.bfloat16, gen, scale=2.0)
        if step:
            ref.accumulated_attention = {0: dev.accumulated_attention[0].clone()}
        ref.update_attention_scores([ref_probs(q, k)])
        dev.update_from_queries([q], [k])
        check_step(ref, dev, 1, B, K + step, f"step {step}")


def capture_of(queries, keys, masks=None):
    cap = QueryCapture(len(queries))
    for l, (q, k) in enumerate(zip(queries, keys)):
        cap._record(l, q, k, None if masks is None else masks[l], q.size(-1) ** -0.5)
    return cap


def check_topk(scores, rows, k):
    s = scores.float()
    kth = torch.topk(s, k).values[-1]
    kept = torch.zeros_like(s, dtype=torch.bool)
    kept[rows] = True
    assert rows.numel() == k and bool((rows[1:] > rows[:-1]).all())
    assert bool((s[kept] >= kth).all()) and bool(kept[s > kth].all())


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("B,Hkv,G", [(1, 2, 4), (3, 2, 4)])
def test_kept_rows_through_the_function_and_compress_(dtype, B, Hkv, G):
    """h2o_attention_compress(attention_queries=...) and KVSlabCache.compress_: per batch entry the kept middle rows are
    a tie-aware top-k of that entry's device score row, shared by its KV heads; sinks and the recent window kept; the
    two paths bit-equal."""
    dt = DT[dtype]
    L, S, D = 3, 400, 64
    gen = torch.Generator(device="cuda").manual_seed(15 + B)
    k = torch.randn(L, B, Hkv, S, D, generator=gen, device="cuda").to(dt)
    pos = torch.arange(S, device="cuda", dtype=torch.float32)
    v = torch.zeros(B, Hkv, S, D, device="cuda")
    v[..., 0], v[..., 1] = pos // 16, pos % 16
    kv = [(k[l], v.to(dt)) for l in range(L)]
    q = [(2 * torch.randn(B, Hkv * G, 1, D, generator=gen, device="cuda")).to(dt) for _ in range(L)]
    _, m_fn = pair(L, Hkv * G)
    _, m_slab = pair(L, Hkv * G)
    out = kvcompress.h2o_attention_compress(kv, attention_queries=capture_of(q, [k[l] for l in range(L)]),
                                            h2o_manager=m_fn, **KW)
    slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
    slab.compress_("h2o_attention", attention_queries=capture_of(q, [slab[l][0] for l in range(L)]),
                   h2o_manager=m_slab, **KW)
    for l in range(L):
        row = m_fn._score_row(l, B, S - 40 - 4)
        assert torch.equal(row, m_slab._score_row(l, B, S - 40 - 4))
        for b in range(B):
            got = (out[l][1][b, :, :, 0].float() * 16 + out[l][1][b, :, :, 1].float()).long()
            for h in range(1, Hkv):
                assert torch.equal(got[0], got[h])
            assert got[0, :4].tolist() == [0, 1, 2, 3] and got[0, -40:].tolist() == list(range(S - 40, S))
            check_topk(row[b], got[0, 4:-40] - 4, 16)
        assert torch.equal(slab[l][0], out[l][0]) and torch.equal(slab[l][1], out[l][1])


def _tiny(kind):
    from transformers import GPTNeoXConfig, GPTNeoXForCausalLM, LlamaConfig, LlamaForCausalLM

    torch.manual_seed(0)
    if kind == "neox":
        cfg = GPTNeoXConfig(vocab_size=256, hidden_size=256, num_hidden_layers=3, num_attention_heads=4,
                            intermediate_size=256, max_position_embeddings=512, rotary_pct=0.25)
        return GPTNeoXForCausalLM(cfg).eval().cuda()
    cfg = LlamaConfig(vocab_size=256, hidden_size=256, num_hidden_layers=3, num_attention_heads=8,
                      num_key_value_heads=2, intermediate_size=256, max_position_embeddings=512)
    return LlamaForCausalLM(cfg).eval().cuda()


@pytest.mark.parametrize("kind", ["neox", "llama_gqa"])
def test_hf_capture_path_matches_the_eager_path(kind):
    """Prefill, a chunked prefill and 20 decode steps of a tiny fp32 model: the accumulators the capture path builds
    (SDPA, no output_attentions) match the eager output_attentions path's within the fp32 tolerance at every step."""
    from transformers import DynamicCache

    model = _tiny(kind)
    cfg = model.config
    L, Hq = cfg.num_hidden_layers, cfg.num_attention_heads
    ids = torch.randint(0, cfg.vocab_size, (1, 24 + 8 + 20), generator=torch.Generator().manual_seed(5)).cuda()
    args = dict(KW, num_layers=L, num_heads=Hq, decay_factor=0.9)
    by_attn, by_query = H2OScoreSlab(**args), H2OScoreSlab(**args)
    c_eager, c_cap = DynamicCache(), DynamicCache()
    steps = [(0, 24), (24, 32)] + [(p, p + 1) for p in range(32, 52)]
    with torch.inference_mode():
        for a, b in steps:
            model.set_attn_implementation("eager")
            out = model(ids[:, a:b], past_key_values=c_eager, use_cache=True, output_attentions=True)
            by_attn.update_attention_scores(out.attentions)
            with kvcompress.capture_queries(model) as cap:
                model(ids[:, a:b], past_key_values=c_cap, use_cache=True)
            by_query.update_from_queries(cap.queries, cap.keys, cap.masks, cap.scaling)
            for l in range(L):
                assert_close_ulp(by_query.accumulated_attention[l], by_attn.accumulated_attention[l],
                                 f"{kind} step {a}:{b} layer {l}")


@pytest.mark.parametrize("cache", ["dynamic", "slab"])
def test_harness_with_queries_matches_reference_golden(cache):
    """evaluate_with_attention_compression(scores="queries") on both caches: the reference's cache lengths and NLLs
    (harness_golden.json), with the thresholds of the attentions path's golden test."""
    import harness_cases as H
    from kvcompress.evaluate_attention import evaluate_with_attention_compression

    golden = json.load(open(os.path.join(GOLDEN_DIR, "harness_golden.json")))
    want = golden["cases"]["h2o_attention"]
    model, ids = H.tiny_model_and_ids("cuda")
    got = evaluate_with_attention_compression(model, input_ids=ids.cuda(), skip_layers=[], show_progress=False,
                                              return_nlls=True, cache=cache, scores="queries", **H.ATTN_KW)
    assert got["cache_lengths"] == want["lengths"] and got["final_cache_size"] == want["final_cache_size"]
    assert got["num_tokens"] == H.TOKENS - 1
    assert max(abs(a - b) for a, b in zip(got["nlls"], want["nlls"])) < 5e-3
    assert abs(got["perplexity"] / want["perplexity"] - 1) < 1e-3


def test_one_decode_step_is_three_launches_without_aten_or_sync():
    """update_from_queries + compress_ on a slab at steady state: stats, accumulate and compaction launches, no ATen
    kernel in the trace and no synchronising call."""
    L, B, Hq, Hkv, D = 4, 2, 8, 2, 64
    budget = 60
    gen = torch.Generator(device="cuda").manual_seed(6)
    k, v = torch.randn(B, Hkv, budget + 1, D, generator=gen, device="cuda").bfloat16(), \
        torch.randn(B, Hkv, budget + 1, D, generator=gen, device="cuda").bfloat16()
    slab = KVSlabCache.from_legacy_cache([(k, v)] * L, capacity=budget + 8)
    dev = H2OScoreSlab(num_layers=L, num_heads=Hq, **KW)
    q = [torch.randn(B, Hq, 1, D, generator=gen, device="cuda").bfloat16() for _ in range(L)]
    new = [(k[:, :, :1].contiguous(), v[:, :, :1].contiguous())] * L

    def step():
        cap = capture_of(q, [slab[l][0] for l in range(L)])
        dev.update_from_queries(cap.queries, cap.keys, cap.masks, cap.scaling)
        slab.compress_("h2o_attention", h2o_manager=dev, **KW)

    step()                      # warm-up: buffers, workspace, plan caches
    slab.append(new)
    torch.cuda.synchronize()
    n0 = _engine.launch_count()
    torch.cuda.set_sync_debug_mode("error")
    try:
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.set_sync_debug_mode(0)
            torch.cuda.synchronize()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert _engine.launch_count() - n0 == 3
    assert slab.lengths == [budget] * L
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names and all("kvc_" in n for n in names), names
    assert sum("kvc_h2o_qk_stats_kernel" in n for n in names) == 1
    assert sum("kvc_h2o_qk_accumulate_kernel" in n for n in names) == 1
    assert sum("kvc_slab_compress_kernel" in n for n in names) == 1
