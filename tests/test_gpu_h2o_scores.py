"""-m gpu: H2OScoreSlab — the H2O score bookkeeping on the device (kvc_h2o_accumulate) and the compaction ranked by
its head-summed score rows (KVC_SCORE_GIVEN_SCORE_SHARED) — against the torch H2OAttentionManager and the rows the
REAL reference kept (tests/golden/extras_golden.json, harness_golden.json)."""

import json
import os

import pytest
import torch

import kvcompress
from kvcompress import H2OAttentionManager, H2OScoreSlab, KVSlabCache, _engine

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
MANTISSA = {torch.bfloat16: 7, torch.float16: 10}


def attention(B, Hq, Q, K, dtype, gen, sharp=2.0):
    return torch.softmax(sharp * torch.randn(B, Hq, Q, K, generator=gen, device="cuda"), dim=-1).to(dtype)


def assert_close_ulp(got, want, what):
    """16-bit: within one unit in the last place of the larger magnitude; fp32: 1e-5 relative."""
    g, w = got.double(), want.double()
    if got.dtype == torch.float32:
        bound = 1e-5 * torch.maximum(g.abs(), w.abs()) + 1e-30
    else:
        mag = torch.maximum(g.abs(), w.abs()).clamp_min(2.0 ** -24)
        bound = torch.exp2(torch.floor(torch.log2(mag)) - MANTISSA[got.dtype])
    bad = (g - w).abs() > bound
    assert not bool(bad.any()), f"{what}: {int(bad.sum())} entries off, worst {float((g - w).abs().max())}"


def pair(L, Hq, capacity=None):
    args = dict(start_size=4, heavy_hitter_size=16, recent_size=40, num_layers=L, num_heads=Hq, decay_factor=0.9)
    return H2OAttentionManager(**args), H2OScoreSlab(capacity=capacity, **args)


@pytest.mark.parametrize("dtype", ["f32", "bf16", "f16"])
def test_accumulators_bit_identical_for_one_query(dtype):
    """A sequence that grows, repeats a key length, updates the same attentions twice, shrinks (reset), skips layers
    and passes None entries: the device accumulators equal the torch manager's bit for bit (n_query = 1)."""
    dt = DT[dtype]
    L, B, Hq = 4, 2, 6
    ref, dev = pair(L, Hq, capacity=64)  # small capacity: the buffers double on the way
    gen = torch.Generator(device="cuda").manual_seed(1)
    for step, (K, skip, none) in enumerate([(100, [], []), (101, [1], []), (101, [], [2]), (150, [], []),
                                            (150, [0], []), (90, [], []), (91, [3], [1]), (300, [], [])]):
        attn = [None if l in none else attention(B, Hq, 1, K, dt, gen) for l in range(L)]
        repeats = 2 if step == 2 else 1  # the harness updates, then the compress call updates again
        for _ in range(repeats):
            ref.update_attention_scores(attn, skip)
            dev.update_attention_scores(attn, skip)
        assert dev.current_seq_len == ref.current_seq_len
        assert sorted(dev.accumulated_attention) == sorted(ref.accumulated_attention)
        for l, want in ref.accumulated_attention.items():
            got = dev.accumulated_attention[l]
            assert got.shape == want.shape and got.dtype == want.dtype, (step, l)
            assert torch.equal(got, want), (step, l)
    assert dev.capacity >= 300
    dev.reset()
    ref.reset()
    attn = [attention(B, Hq, 1, 120, dt, gen) for _ in range(L)]
    ref.update_attention_scores(attn)
    dev.update_attention_scores(attn)
    for l in range(L):
        assert torch.equal(dev.accumulated_attention[l], ref.accumulated_attention[l])


@pytest.mark.parametrize("dtype", ["f32", "bf16", "f16"])
@pytest.mark.parametrize("Q,K", [(7, 300), (128, 264), (264, 264)])
def test_accumulators_and_score_rows_for_many_queries(dtype, Q, K):
    """n_query > 1 (prefill-sized up to n_query = key_len; aligned and unaligned rows): every update step agrees with
    the torch manager's step from the same state within 1 ulp / 1e-5, and the score row with the head sum of the
    accumulators."""
    dt = DT[dtype]
    L, B, Hq = 2, 2, 4
    ref, dev = pair(L, Hq)
    gen = torch.Generator(device="cuda").manual_seed(2 + Q)
    for step in range(2):
        attn = [attention(B, Hq, Q, K, dt, gen, sharp=3.0) for _ in range(L)]
        if step:  # start the torch step from the device's state, so that one step's rounding is compared
            ref.accumulated_attention = {l: dev.accumulated_attention[l].clone() for l in range(L)}
        ref.update_attention_scores(attn)
        dev.update_attention_scores(attn)
        for l in range(L):
            acc = dev.accumulated_attention[l]
            assert_close_ulp(acc, ref.accumulated_attention[l], f"acc step {step} layer {l}")
            lo, hi = 4, K - 40
            row = dev._score_row(l, B, hi - lo)
            assert_close_ulp(row, acc[:, :, lo:hi].sum(dim=1), f"score step {step} layer {l}")


def check_topk(scores, rows, k):
    """`rows` (ascending, relative) is a valid top-k of `scores` with ties: everything strictly above the k-th value is
    kept, nothing below it."""
    s = scores.float()
    kth = torch.topk(s, k).values[-1]
    kept = torch.zeros_like(s, dtype=torch.bool)
    kept[rows] = True
    assert rows.numel() == k and bool((rows[1:] > rows[:-1]).all())
    assert bool((s[kept] >= kth).all()) and bool(kept[s > kth].all())


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_kept_rows_are_a_top_k_of_the_device_score_row(dtype):
    """Through h2o_attention_compress and KVSlabCache.compress_: per batch entry the kept middle rows are a tie-aware
    top-k of that entry's own score row, identical across its KV heads; the sinks and the recent window are kept."""
    dt = DT[dtype]
    L, B, Hq, Hkv, S, D = 3, 3, 8, 2, 400, 64
    _, dev = pair(L, Hq)
    gen = torch.Generator(device="cuda").manual_seed(5)
    attn = [attention(B, Hq, 1, S, dt, gen) for _ in range(L)]
    k = torch.randn(L, B, Hkv, S, D, generator=gen, device="cuda").to(dt)
    pos = torch.arange(S, device="cuda", dtype=torch.float32)
    v = torch.zeros(B, Hkv, S, D, device="cuda")
    v[..., 0], v[..., 1] = pos // 16, pos % 16   # the row position, in values every dtype holds exactly
    kv = [(k[l], v.to(dt)) for l in range(L)]
    kw = dict(start_size=4, heavy_hitter_size=16, recent_size=40)
    out = kvcompress.h2o_attention_compress(kv, attention_scores=attn, h2o_manager=dev, **kw)
    slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
    slab.compress_("h2o_attention", h2o_manager=dev, **kw)   # the accumulators as they are (no second update)
    for l in range(L):
        row = dev._score_row(l, B, S - 40 - 4)
        for b in range(B):
            got = (out[l][1][b, :, :, 0].float() * 16 + out[l][1][b, :, :, 1].float()).long()
            assert torch.equal(got[0], got[1]), "heads of one batch entry share their heavy hitters"
            assert got[0, :4].tolist() == [0, 1, 2, 3] and got[0, -40:].tolist() == list(range(S - 40, S))
            check_topk(row[b], got[0, 4:-40] - 4, 16)
        assert torch.equal(slab[l][0], out[l][0]) and torch.equal(slab[l][1], out[l][1])


def test_reference_golden_rows_function_and_slab():
    """The REAL reference's kept rows (extras_golden.json "h2o": a decode sequence that shrinks the cache, a skipped
    layer) through both the function and the in-place path; K and V bit-equal to the torch-manager path."""
    import extras_cases as E

    want = json.load(open(os.path.join(GOLDEN_DIR, "extras_golden.json")))
    c = E.H2O_CASE
    kw = dict(start_size=c["start_size"], heavy_hitter_size=c["heavy_hitter_size"], recent_size=c["recent_size"],
              skip_layers=c["skip_layers"])
    mk = dict(start_size=c["start_size"], heavy_hitter_size=c["heavy_hitter_size"], recent_size=c["recent_size"],
              num_layers=c["layers"], num_heads=c["heads"], decay_factor=c["decay_factor"])
    m_torch, m_fn, m_slab = H2OAttentionManager(**mk), H2OScoreSlab(**mk), H2OScoreSlab(**mk)
    for step, ref in enumerate(want["h2o"]):
        kv, attn = E.h2o_inputs(step, ref["seq_len"])
        kv = [(k.cuda(), v.cuda()) for k, v in kv]
        attn = [a.cuda() for a in attn]
        base = kvcompress.h2o_attention_compress(kv, attention_scores=attn, h2o_manager=m_torch, **kw)
        out = kvcompress.h2o_attention_compress(kv, attention_scores=attn, h2o_manager=m_fn, **kw)
        slab = KVSlabCache.from_legacy_cache(kv, capacity=ref["seq_len"] + 4)
        slab.compress_("h2o_attention", attention_scores=attn, h2o_manager=m_slab, **kw)
        assert [k.size(2) for k, _ in out] == ref["lengths"] and slab.lengths == ref["lengths"], step
        for l in range(len(kv)):
            assert out[l][1][0, :, :, 0].long().tolist() == ref["rows"][l], (step, l)
            assert torch.equal(out[l][0], base[l][0]) and torch.equal(out[l][1], base[l][1]), (step, l)
            assert torch.equal(slab[l][0], base[l][0]) and torch.equal(slab[l][1], base[l][1]), (step, l)


@pytest.mark.parametrize("B,Hq,Hkv", [(1, 8, 2), (3, 4, 4), (3, 8, 2)])
def test_gqa_and_batches_keep_what_the_torch_path_keeps_per_entry(B, Hq, Hkv):
    """Each batch entry keeps the rows the torch manager + function keep on that entry alone (the torch manager
    refuses batch > 1); GQA sums the mass of all Hq query heads."""
    L, S, D = 2, 300, 32
    gen = torch.Generator(device="cuda").manual_seed(B * 10 + Hq)
    kw = dict(start_size=4, heavy_hitter_size=16, recent_size=40)
    mk = dict(kw, num_layers=L, num_heads=Hq, decay_factor=0.9)
    dev = H2OScoreSlab(**mk)
    steps = []
    for step, K in enumerate((S - 1, S)):  # two updates: the second one decays the first
        steps.append([attention(B, Hq, 1, K, torch.float32, gen) for _ in range(L)])
    kv = [(torch.randn(B, Hkv, S, D, generator=gen, device="cuda"),
           torch.arange(S, device="cuda", dtype=torch.float32).view(1, 1, S, 1).expand(B, Hkv, S, D).contiguous())
          for _ in range(L)]
    dev.update_attention_scores(steps[0])
    out = kvcompress.h2o_attention_compress(kv, attention_scores=steps[1], h2o_manager=dev, **kw)
    for b in range(B):
        ref = H2OAttentionManager(**mk)
        ref.update_attention_scores([a[b:b + 1] for a in steps[0]])
        want = kvcompress.h2o_attention_compress([(k[b:b + 1], v[b:b + 1]) for k, v in kv],
                                                 attention_scores=[a[b:b + 1] for a in steps[1]], h2o_manager=ref, **kw)
        for l in range(L):
            assert torch.equal(out[l][0][b:b + 1], want[l][0]) and torch.equal(out[l][1][b:b + 1], want[l][1]), (b, l)


def test_heavy_hitter_indices_match_the_torch_manager():
    L, Hq, K = 2, 4, 200
    ref, dev = pair(L, Hq)
    assert torch.equal(dev.get_heavy_hitter_indices(0, K), ref.get_heavy_hitter_indices(0, K))  # no data: spaced
    gen = torch.Generator(device="cuda").manual_seed(9)
    attn = [attention(1, Hq, 1, K, torch.float32, gen) for _ in range(L)]
    ref.update_attention_scores(attn)
    dev.update_attention_scores(attn)
    for seq_len in (K, K - 30, K + 50, 44):  # the update's region, a shorter cache (re-score), a longer one, empty
        got, want = dev.get_heavy_hitter_indices(1, seq_len), ref.get_heavy_hitter_indices(1, seq_len)
        assert got.dim() == want.dim() == 1 and got.dtype == want.dtype
        assert torch.equal(got.cpu(), want.cpu()), seq_len


def test_attention_dtype_must_match_the_cache():
    _, dev = pair(1, 2)
    gen = torch.Generator(device="cuda").manual_seed(4)
    dev.update_attention_scores([attention(1, 2, 1, 100, torch.float32, gen)])
    kv = [(torch.randn(1, 2, 100, 16, device="cuda").bfloat16(), torch.randn(1, 2, 100, 16, device="cuda").bfloat16())]
    with pytest.raises(ValueError, match="float32.*bfloat16"):
        kvcompress.h2o_attention_compress(kv, h2o_manager=dev, start_size=4, heavy_hitter_size=16, recent_size=40)


@pytest.mark.parametrize("cache", ["dynamic", "slab"])
def test_harness_matches_reference_golden(cache):
    """evaluate_with_attention_compression with an H2OScoreSlab, on the DynamicCache and on the slab: the reference's
    cache lengths and NLLs (harness_golden.json, produced with the REAL reference on CPU)."""
    import harness_cases as H
    from kvcompress.evaluate_attention import evaluate_with_attention_compression

    golden = json.load(open(os.path.join(GOLDEN_DIR, "harness_golden.json")))
    want = golden["cases"]["h2o_attention"]
    model, ids = H.tiny_model_and_ids("cuda", attn_implementation="eager")
    manager = H2OScoreSlab(num_layers=H.MODEL_KW["num_hidden_layers"], num_heads=H.MODEL_KW["num_attention_heads"],
                           **H.ATTN_KW)
    got = evaluate_with_attention_compression(model, input_ids=ids.cuda(), h2o_manager=manager, skip_layers=[],
                                              show_progress=False, return_nlls=True, cache=cache, **H.ATTN_KW)
    assert got["cache_lengths"] == want["lengths"] and got["final_cache_size"] == want["final_cache_size"]
    assert got["num_tokens"] == H.TOKENS - 1
    assert max(abs(a - b) for a, b in zip(got["nlls"], want["nlls"])) < 5e-3
    assert abs(got["perplexity"] / want["perplexity"] - 1) < 1e-3


def test_one_decode_step_is_two_launches_without_aten_or_sync():
    """Update + compress_ on a slab at steady state: one accumulate launch, one compaction launch, no ATen kernel in
    the trace and no synchronising call."""
    L, B, Hq, Hkv, D = 4, 2, 8, 2, 64
    kw = dict(start_size=4, heavy_hitter_size=16, recent_size=40)
    budget = 60
    gen = torch.Generator(device="cuda").manual_seed(6)
    k, v = torch.randn(B, Hkv, budget + 1, D, generator=gen, device="cuda").bfloat16(), \
        torch.randn(B, Hkv, budget + 1, D, generator=gen, device="cuda").bfloat16()
    slab = KVSlabCache.from_legacy_cache([(k, v)] * L, capacity=budget + 8)
    dev = H2OScoreSlab(num_layers=L, num_heads=Hq, **kw)
    attn = [attention(B, Hq, 1, budget + 1, torch.bfloat16, gen) for _ in range(L)]
    new = [(k[:, :, :1].contiguous(), v[:, :, :1].contiguous())] * L

    def step():
        dev.update_attention_scores(attn)
        slab.compress_("h2o_attention", h2o_manager=dev, **kw)

    step()                      # warm-up: buffers, plan caches
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
    assert _engine.launch_count() - n0 == 2
    assert slab.lengths == [budget] * L
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names and all("kvc_" in n for n in names), names
    assert sum("kvc_h2o_accumulate_kernel" in n for n in names) == 1
    assert sum("kvc_slab_compress_kernel" in n for n in names) == 1
