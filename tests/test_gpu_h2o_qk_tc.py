"""-m gpu: H2OScoreSlab(tensor_cores=True) — the H2O query update on the tensor cores (kvc_h2o_accumulate_qk_tc) —
against fp64 torch logits -> softmax -> .to(dtype) -> the torch manager's update, against the CUDA-core form
(kvc_h2o_accumulate_qk) at prompt scale and on captured HF queries, through both compress paths, and as a decode step."""

import pytest
import torch

import kvcompress
from kvcompress import H2OAttentionManager, H2OScoreSlab, KVSlabCache, QueryCapture, _engine

pytestmark = pytest.mark.gpu

DT = {"bf16": torch.bfloat16, "f16": torch.float16}
MANTISSA = {torch.bfloat16: 7, torch.float16: 10}
KW = dict(start_size=4, heavy_hitter_size=16, recent_size=40)


def assert_close_ulp(got, want, what, scale=1):
    """Within one unit in the last place of the larger magnitude, except at rounding near-ties: a probability whose
    fp32 value lies within ~1e-6 of a rounding boundary of the dtype can round the other way than the reference's,
    which moves the mass by one ulp of that probability, and the update's own rounding of round(acc * decay) + mass can
    then land one more ulp away.  So at most 2 ulps anywhere, and beyond 1 ulp on at most 0.1% of the entries (both
    ulp counts times `scale`)."""
    g, w = got.double(), want.double()
    mag = torch.maximum(g.abs(), w.abs()).clamp_min(2.0 ** -14 if got.dtype == torch.float16 else 2.0 ** -126)
    ulp = torch.exp2(torch.floor(torch.log2(mag)) - MANTISSA[got.dtype])
    diff = (g - w).abs()
    assert not bool((diff > 2 * scale * ulp).any()), f"{what}: {int((diff > 2 * scale * ulp).sum())} entries beyond " \
                                                     f"{2 * scale} ulps"
    n1 = int((diff > scale * ulp).sum())
    assert n1 <= max(1, diff.numel() // 1000), f"{what}: {n1} of {diff.numel()} entries beyond {scale} ulp"


def ref_probs(q, k, mask=None, scaling=None):
    """The contract in fp64, one query head at a time: logits, visibility (mask or causal), softmax, 0 where invisible,
    then .to(dtype)."""
    B, Hq, T, D = q.shape
    S, G = k.size(2), Hq // k.size(1)
    scaling = D ** -0.5 if scaling is None else scaling
    if mask is None:
        vis = (torch.arange(S, device=q.device).view(1, S) <=
               (S - T + torch.arange(T, device=q.device)).view(T, 1)).view(1, T, S)
    else:
        vis = (mask[:, 0] if mask.dim() == 4 else mask)[..., :S]
    out = torch.empty(B, Hq, T, S, dtype=q.dtype, device=q.device)
    for h in range(Hq):
        s = scaling * torch.matmul(q[:, h].double(), k[:, h // G].double().transpose(-1, -2))
        p = torch.softmax(s.masked_fill(~vis, float("-inf")), dim=-1).nan_to_num(0.0)
        out[:, h] = p.masked_fill(~vis, 0.0).to(q.dtype)
    return out


def inputs(B, Hkv, G, T, K, D, dtype, gen, cap_extra=24, scale=2.0):
    """Queries and keys; the keys are a strided view [B, Hkv, K, D] of a longer slab-like buffer."""
    q = (scale * torch.randn(B, Hkv * G, T, D, generator=gen, device="cuda")).to(dtype)
    kbuf = torch.randn(B, Hkv, K + cap_extra, D, generator=gen, device="cuda").to(dtype)
    return q, kbuf[:, :, :K]


def managers(L, Hq, **kw):
    args = dict(KW, num_layers=L, num_heads=Hq, decay_factor=0.9)
    return H2OAttentionManager(**args), H2OScoreSlab(tensor_cores=True, **args, **kw)


def check_step(ref, dev, L, B, K, what):
    for l in range(L):
        acc = dev.accumulated_attention[l]
        assert_close_ulp(acc, ref.accumulated_attention[l], f"{what} acc layer {l}")
        lo, hi = KW["start_size"], K - KW["recent_size"]
        if hi > lo:
            assert_close_ulp(dev._score_row(l, B, hi - lo), acc[:, :, lo:hi].sum(dim=1), f"{what} score layer {l}")


def run_against_reference(dtype, G, T, K, D, B, Hkv, L, seed, masks=None):
    ref, dev = managers(L, Hkv * G)
    gen = torch.Generator(device="cuda").manual_seed(seed)
    for step in range(2):
        Ks = K + step * min(T, 5)   # the second step grows the cache (and decays the first step's mass)
        Ts = min(T, Ks)
        qk = [inputs(B, Hkv, G, Ts, Ks, D, dtype, gen) for _ in range(L)]
        if step:
            ref.accumulated_attention = {l: dev.accumulated_attention[l].clone() for l in range(L)}
        ref.update_attention_scores([ref_probs(q, k) for q, k in qk])
        dev.update_from_queries([q for q, _ in qk], [k for _, k in qk])
        assert dev.current_seq_len == Ks
        check_step(ref, dev, L, B, Ks, f"step {step}")


@pytest.mark.parametrize("dtype", ["bf16", "f16"])
@pytest.mark.parametrize("G", [1, 4, 8])
@pytest.mark.parametrize("D", [64, 80, 128])
@pytest.mark.parametrize("T,K", [(1, 517), (7, 300), (128, 333), (1000, 1000), (4096, 4096)])
def test_accumulators_and_score_rows_match_the_reference(dtype, G, D, T, K):
    """Two steps from the device's state: the accumulators and the score row within the ulp bound of fp64 logits ->
    softmax -> .to(dtype) -> the torch manager's update."""
    big = T * K > 1 << 20
    run_against_reference(DT[dtype], G, T, K, D, B=1 if big else 2, Hkv=1 if big else 2, L=1 if big else 2,
                          seed=G * 1000 + T + K + D)


def test_long_keys():
    """B 1, Hq 32, Hkv 8, D 128, 256 queries over 32768 keys (bf16), two steps."""
    run_against_reference(torch.bfloat16, 4, 256, 32768, 128, B=1, Hkv=8, L=1, seed=14)


@pytest.mark.parametrize("form", ["4d", "3d"])
def test_masks_and_the_causal_rule(form):
    """Bool masks [B, 1, T, K] and [B, T, K]: left padding gets exactly 0, a query row that sees nothing adds nothing,
    a causal mask gives the bits of the causal rule."""
    L, B, Hkv, G, T, K, D = 1, 3, 2, 4, 150, 700, 128
    gen = torch.Generator(device="cuda").manual_seed(12)
    q, k = inputs(B, Hkv, G, T, K, D, torch.bfloat16, gen)
    mask = torch.ones(B, 1, T, K, dtype=torch.bool, device="cuda")
    mask[0, :, :, :30] = False            # entry 0: 30 left-padded key columns
    mask[1, :, 2, :] = False              # entry 1: query 2 sees nothing
    mask[2] = torch.tril(torch.ones(T, K, dtype=torch.bool, device="cuda"), diagonal=K - T)
    m = mask if form == "4d" else mask[:, 0]
    ref, dev = managers(L, Hkv * G)
    ref.update_attention_scores([ref_probs(q, k, m)])
    dev.update_from_queries([q], [k], masks=[m])
    acc = dev.accumulated_attention[0]
    assert bool((acc[0, :, :30] == 0).all())
    check_step(ref, dev, L, B, K, "mask")
    keep = [t for t in range(T) if t != 2]
    _, alone = managers(L, Hkv * G)
    alone.update_from_queries([q[1:2, :, keep]], [k[1:2]], masks=[m[1:2, :, keep] if form == "4d" else m[1:2, keep]])
    assert torch.equal(alone.accumulated_attention[0][0], acc[1])
    _, causal = managers(L, Hkv * G)
    causal.update_from_queries([q[2:3]], [k[2:3]])
    assert torch.equal(causal.accumulated_attention[0][0], acc[2])


def test_determinism_and_independence_from_the_launch():
    """The same inputs give the same bits; a layer alone equals the same layer inside a multi-layer launch with other
    shapes; a batch entry alone equals the same entry inside a batch."""
    B, Hkv, G, D = 3, 2, 4, 128
    gen = torch.Generator(device="cuda").manual_seed(13)
    shapes = [(7, 900), (1, 4000), (333, 700), (1024, 1024)]
    L = len(shapes)
    qk = [inputs(B, Hkv, G, T, K, D, torch.bfloat16, gen) for T, K in shapes]
    _, a = managers(L, Hkv * G)
    _, b = managers(L, Hkv * G)
    a.update_from_queries([q for q, _ in qk], [k for _, k in qk])
    b.update_from_queries([q for q, _ in qk], [k for _, k in qk])
    for l in range(L):
        assert torch.equal(a.accumulated_attention[l], b.accumulated_attention[l])
        region = shapes[l][1] - KW["recent_size"] - KW["start_size"]
        assert torch.equal(a._score_row(l, B, region), b._score_row(l, B, region))
    for l in range(L):
        _, one = managers(L, Hkv * G)
        one.update_from_queries([q if i == l else None for i, (q, _) in enumerate(qk)], [k for _, k in qk])
        assert torch.equal(one.accumulated_attention[l], a.accumulated_attention[l]), l
        _, entry = managers(L, Hkv * G)
        entry.update_from_queries([q[1:2] if i == l else None for i, (q, _) in enumerate(qk)], [k[1:2] for _, k in qk])
        assert torch.equal(entry.accumulated_attention[l][0], a.accumulated_attention[l][1]), l


def test_non_contiguous_queries_are_copied_and_give_the_same_bits():
    """q views a tensor map cannot describe (a size-1 position dimension with an odd stride) are copied first."""
    B, Hkv, G, D, K = 2, 2, 4, 80, 400
    gen = torch.Generator(device="cuda").manual_seed(16)
    q, k = inputs(B, Hkv, G, 1, K, D, torch.float16, gen)
    odd = q.as_strided(q.shape, (Hkv * G * D, D, 3, 1))
    assert not _engine._rows_ok(odd)
    _, a = managers(1, Hkv * G)
    _, b = managers(1, Hkv * G)
    a.update_from_queries([q], [k])
    b.update_from_queries([odd], [k])
    assert torch.equal(a.accumulated_attention[0], b.accumulated_attention[0])


def test_prompt_scale_agrees_with_the_cuda_core_form():
    """T = key_len = 16384, one layer, Hkv 1, G 4, D 128, bf16: within twice the bound of the CUDA-core result."""
    B, Hkv, G, T, D = 1, 1, 4, 16384, 128
    gen = torch.Generator(device="cuda").manual_seed(17)
    q, k = inputs(B, Hkv, G, T, T, D, torch.bfloat16, gen)
    args = dict(KW, num_layers=1, num_heads=Hkv * G, decay_factor=0.9)
    tc, cc = H2OScoreSlab(tensor_cores=True, **args), H2OScoreSlab(**args)
    tc.update_from_queries([q], [k])
    cc.update_from_queries([q], [k])
    assert_close_ulp(tc.accumulated_attention[0], cc.accumulated_attention[0], "16384 acc", scale=2)
    lo, hi = KW["start_size"], T - KW["recent_size"]
    assert_close_ulp(tc._score_row(0, B, hi - lo), cc._score_row(0, B, hi - lo), "16384 score", scale=2)


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


@pytest.mark.parametrize("carry", [False, True])
def test_kept_rows_of_compress_are_the_top_k_of_the_managers_score_row(carry):
    """compress_("h2o_attention", attention_queries=...) with a tensor-core manager: per batch entry the kept middle rows
    are a tie-aware top-k of the score row that manager builds from those queries (read from a twin manager fed the
    same queries: the bits are deterministic), shared by the KV heads; sinks and the recent window kept."""
    L, B, Hkv, G, S, D = 3, 2, 2, 4, 400, 128
    gen = torch.Generator(device="cuda").manual_seed(18)
    k = torch.randn(L, B, Hkv, S, D, generator=gen, device="cuda").bfloat16()
    pos = torch.arange(S, device="cuda", dtype=torch.float32)
    v = torch.zeros(B, Hkv, S, D, device="cuda")
    v[..., 0], v[..., 1] = pos // 16, pos % 16
    kv = [(k[l], v.bfloat16()) for l in range(L)]
    q = [(2 * torch.randn(B, Hkv * G, 64, D, generator=gen, device="cuda")).bfloat16() for _ in range(L)]
    _, m = managers(L, Hkv * G, carry_scores=carry)
    _, twin = managers(L, Hkv * G, carry_scores=carry)
    slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
    twin.update_from_queries(q, [slab[l][0] for l in range(L)])
    slab.compress_("h2o_attention", attention_queries=capture_of(q, [slab[l][0] for l in range(L)]), h2o_manager=m,
                   **KW)
    for l in range(L):
        row = twin._score_row(l, B, S - 40 - 4)
        for b in range(B):
            got = (slab[l][1][b, :, :, 0].float() * 16 + slab[l][1][b, :, :, 1].float()).long()
            for h in range(1, Hkv):
                assert torch.equal(got[0], got[h])
            assert got[0, :4].tolist() == [0, 1, 2, 3] and got[0, -40:].tolist() == list(range(S - 40, S))
            check_topk(row[b], got[0, 4:-40] - 4, 16)
            if carry:  # the accumulators moved with their rows
                src = got[0]
                assert torch.equal(m.accumulated_attention[l][b], twin.accumulated_attention[l][b][:, src])


def _tiny(kind):
    from transformers import GPTNeoXConfig, GPTNeoXForCausalLM, LlamaConfig, LlamaForCausalLM

    torch.manual_seed(0)
    if kind == "neox":  # head_dim 80
        cfg = GPTNeoXConfig(vocab_size=256, hidden_size=320, num_hidden_layers=3, num_attention_heads=4,
                            intermediate_size=256, max_position_embeddings=512, rotary_pct=0.25)
        return GPTNeoXForCausalLM(cfg).eval().cuda().bfloat16()
    cfg = LlamaConfig(vocab_size=256, hidden_size=512, num_hidden_layers=3, num_attention_heads=8,  # head_dim 64, GQA
                      num_key_value_heads=2, intermediate_size=256, max_position_embeddings=512)
    return LlamaForCausalLM(cfg).eval().cuda().bfloat16()


@pytest.mark.parametrize("kind", ["neox", "llama_gqa"])
def test_hf_capture_matches_the_cuda_core_form(kind):
    """Prefill, a chunked prefill and 20 decode steps of a tiny bf16 model under capture_queries: the tensor-core
    manager's accumulators stay within the bound of the CUDA-core manager's on the same captured q and K."""
    from transformers import DynamicCache

    model = _tiny(kind)
    cfg = model.config
    L, Hq = cfg.num_hidden_layers, cfg.num_attention_heads
    ids = torch.randint(0, cfg.vocab_size, (1, 200 + 64 + 20), generator=torch.Generator().manual_seed(5)).cuda()
    args = dict(KW, num_layers=L, num_heads=Hq, decay_factor=0.9)
    tc, cc = H2OScoreSlab(tensor_cores=True, **args), H2OScoreSlab(**args)
    cache = DynamicCache()
    steps = [(0, 200), (200, 264)] + [(p, p + 1) for p in range(264, 284)]
    with torch.inference_mode():
        for a, b in steps:
            with kvcompress.capture_queries(model) as cap:
                model(ids[:, a:b], past_key_values=cache, use_cache=True)
            tc.update_from_queries(cap.queries, cap.keys, cap.masks, cap.scaling)
            cc.update_from_queries(cap.queries, cap.keys, cap.masks, cap.scaling)
            for l in range(L):
                assert_close_ulp(tc.accumulated_attention[l], cc.accumulated_attention[l], f"{kind} {a}:{b} layer {l}")


def test_one_decode_step_is_four_launches_without_aten_or_sync():
    """update_from_queries + compress_ on a slab at steady state with a tensor-core manager: the statistics, column-sum,
    score-row and compaction launches, no ATen kernel in the trace and no synchronising call."""
    L, B, Hq, Hkv, D = 4, 2, 8, 2, 64
    budget = 60
    gen = torch.Generator(device="cuda").manual_seed(6)
    k, v = torch.randn(B, Hkv, budget + 1, D, generator=gen, device="cuda").bfloat16(), \
        torch.randn(B, Hkv, budget + 1, D, generator=gen, device="cuda").bfloat16()
    slab = KVSlabCache.from_legacy_cache([(k, v)] * L, capacity=budget + 8)
    dev = H2OScoreSlab(num_layers=L, num_heads=Hq, tensor_cores=True, **KW)
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
    assert _engine.launch_count() - n0 == 4
    assert slab.lengths == [budget] * L
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names and all("kvc_" in n for n in names), names
    assert sum("kvc_h2o_tc_kernel" in n for n in names) == 2
    assert sum("kvc_h2o_accumulate_kernel" in n for n in names) == 1
    assert sum("kvc_slab_compress_kernel" in n for n in names) == 1
