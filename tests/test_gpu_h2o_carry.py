"""-m gpu: cumulative H2O — per-row state carried through the compaction (kvc_slab_compress_carry,
kvc_compress_layers_carry) and H2OScoreSlab(carry_scores=True) against torch loops that gather the accumulators with
the kept rows."""

import json
import os

import pytest
import torch

import kvcompress
from kvcompress import H2OScoreSlab, KVSlabCache, _engine
from kvcompress import _planner as P
from kvcompress.utils import normalize_kv_cache, to_dynamic_cache

from test_gpu_h2o_queries import assert_close_ulp, capture_of, ref_probs

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DT = {"f32": torch.float32, "bf16": torch.bfloat16, "f16": torch.float16}
KW = dict(start_size=4, heavy_hitter_size=16, recent_size=40)
BUDGET = 60


def expect_carried(acc, idx, group, prev_len):
    """acc'[b, h*G+g, i] = acc[b, h*G+g, idx[b, h, i]] where idx < prev_len, 0 elsewhere."""
    src = idx.long().repeat_interleave(group, dim=1)
    want = acc.gather(-1, src)
    return torch.where(src < prev_len, want, torch.zeros_like(want))


# ---------------------------------------------------------------------------------------------- 1. carry exactness
def _plans(S, kind):
    if kind == "h2o":
        return P.plan_h2o([S], 4, 32, 40, skip_layers=())
    if kind == "workspace":                   # l2_compress keep 0.8 of 32K rows: keys / kept indices in the workspace
        return P.plan_l2([S], 0.8, 0, skip_layers=())
    return [P.LayerPlan(P.GATHER, S, sink=S)]  # "still": every row stays where it is


CASES = [  # dtype, G, B, D (compiled and generic row widths), S, plan kind, prev_len
    ("f32", 1, 1, 64, 300, "h2o", 300),
    ("f32", 4, 3, 24, 300, "h2o", 250),
    ("bf16", 8, 1, 128, 517, "h2o", 517),
    ("bf16", 4, 3, 48, 400, "h2o", 330),
    ("f16", 4, 1, 64, 300, "h2o", 299),
    ("f16", 1, 3, 80, 300, "h2o", 1000),
    ("f32", 4, 1, 64, 32768, "workspace", 30000),
    ("bf16", 4, 3, 64, 200, "still", 150),
    ("f32", 1, 1, 24, 200, "still", 200),
]


@pytest.mark.parametrize("dtype,G,B,D,S,kind,prev_len", CASES)
def test_carry_is_exact_on_both_paths(dtype, G, B, D, S, kind, prev_len):
    """Both entry points: acc'[..., :C] is acc gathered with the kept rows (per query head of the KV head), bit for
    bit, with zeros where src >= prev_len; K, V, norms and idx_out are byte-identical to the call without carry."""
    dt, H = DT[dtype], 2
    gen = torch.Generator(device="cuda").manual_seed(S + G * 10 + B)
    k = torch.randn(B, H, S, D, generator=gen, device="cuda").to(dt)
    v = torch.randn(B, H, S, D, generator=gen, device="cuda").to(dt)
    acc0 = torch.randn(B, H * G, S + 7, generator=gen, device="cuda").to(dt)
    plans = _plans(S, kind)
    C = plans[0].out_len
    if kind == "workspace":
        shape = _engine._SHAPE.pack(B, H, D, _engine.KVC_DTYPE[dt], torch.cuda.current_device())
        recs = b"".join(_engine._PLAN.pack(p.seq_len, p.sink, p.sel_lo, p.sel_hi, p.k_sel, p.tail, p.score,
                                           p.pool_kernel) for p in plans)
        assert _engine.load_library().kvc_workspace_bytes(shape, 1, recs) > 0
    # function path: K / V out of place, acc in place
    acc = acc0.clone()
    plain, idx = _engine.run_plans([(k, v)], plans, return_indices=True)
    out, idx_c = _engine.run_plans([(k, v)], plans, return_indices=True, carry={0: (acc, G, prev_len)})
    assert torch.equal(idx[0], idx_c[0])
    assert torch.equal(out[0][0], plain[0][0]) and torch.equal(out[0][1], plain[0][1])
    assert torch.equal(acc[..., :C], expect_carried(acc0, idx[0], G, min(prev_len, S)))
    assert torch.equal(acc[..., C:], acc0[..., C:]) or kind != "still"
    # slab path: everything in place
    slab_a = KVSlabCache.from_legacy_cache([(k, v)], capacity=S + 8)
    slab_b = KVSlabCache.from_legacy_cache([(k, v)], capacity=S + 8)
    acc = acc0.clone()
    _, sidx = slab_a.apply_plans_(plans, return_indices=True)
    _, sidx_c = slab_b.apply_plans_(plans, return_indices=True, carry={0: (acc, G, prev_len)})
    assert torch.equal(sidx[0], sidx_c[0])
    assert slab_b.lengths == slab_a.lengths == [C]
    assert torch.equal(slab_a[0][0], slab_b[0][0]) and torch.equal(slab_a[0][1], slab_b[0][1])
    assert torch.equal(slab_a.key_norms(0), slab_b.key_norms(0))
    assert torch.equal(acc[..., :C], expect_carried(acc0, sidx[0], G, min(prev_len, S)))
    if kind == "h2o":  # the two paths keep the same rows here (norms from the same rows)
        assert torch.equal(sidx[0], idx[0])


def test_carry_of_several_layers_in_one_launch_and_layers_without_acc():
    """Layers with and without carried state in one launch: only the carried layers' acc changes."""
    B, H, G, D, S = 2, 2, 4, 64, 300
    gen = torch.Generator(device="cuda").manual_seed(3)
    kv = [(torch.randn(B, H, S, D, generator=gen, device="cuda").bfloat16(),
           torch.randn(B, H, S, D, generator=gen, device="cuda").bfloat16()) for _ in range(3)]
    acc0 = torch.randn(3, B, H * G, S, generator=gen, device="cuda").bfloat16()
    acc = acc0.clone()
    plans = P.plan_h2o([S] * 3, 4, 32, 40, skip_layers=())
    n0 = _engine.launch_count()
    _, idx = _engine.run_plans(kv, plans, return_indices=True, carry={0: (acc[0], G, S), 2: (acc[2], G, 200)})
    assert _engine.launch_count() - n0 == 1
    C = plans[0].out_len
    assert torch.equal(acc[0, ..., :C], expect_carried(acc0[0], idx[0], G, S))
    assert torch.equal(acc[1], acc0[1])
    assert torch.equal(acc[2, ..., :C], expect_carried(acc0[2], idx[2], G, 200))


# ---------------------------------------------------------------------------------------------- 2. cumulative loop
def _check_topk(scores, rows, k):
    s = scores.float()
    kth = torch.topk(s, k).values[-1]
    kept = torch.zeros_like(s, dtype=torch.bool)
    kept[rows] = True
    assert rows.numel() == k and bool((rows[1:] > rows[:-1]).all())
    assert bool((s[kept] >= kth).all()) and bool(kept[s > kth].all())


def _head_sum(acc, lo, hi):
    """The score row as the device forms it: fp32 sum over the query heads in ascending order, rounded once."""
    s = acc[:, 0, lo:hi].float()
    for h in range(1, acc.size(1)):
        s = s + acc[:, h, lo:hi].float()
    return s.to(acc.dtype)


def _rows(gen, L, B, Hkv, D, n, t0, dt):
    """New K / V rows; V's first two channels encode the token position (exact in every dtype), so that the function
    path's and the slab path's caches are equal only if both keep the same tokens."""
    k = torch.randn(L, B, Hkv, n, D, generator=gen, device="cuda").to(dt)
    v = torch.randn(L, B, Hkv, n, D, generator=gen, device="cuda")
    pos = torch.arange(t0, t0 + n, device="cuda", dtype=torch.float32)
    v[..., 0], v[..., 1] = pos // 64, pos % 64
    return k, v.to(dt)


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
@pytest.mark.parametrize("B,Hkv,G", [(1, 2, 1), (3, 2, 4)])
def test_cumulative_loop_matches_torch(dtype, B, Hkv, G):
    """45 decode steps past the budget, one query per step: after every compaction the device accumulators equal, bit
    for bit, a torch loop acc = round(round(acc * decay) + attn.sum(2)) (zero-extended), acc = acc.gather(-1, kept),
    fed the device's kept rows; every selection is a tie-valid top-k of the torch head-summed scores; the function
    path and the slab path agree bit for bit."""
    dt = DT[dtype]
    L, D, Hq = 2, 64, Hkv * G
    gen = torch.Generator(device="cuda").manual_seed(100 + B * 10 + G)
    args = dict(KW, num_layers=L, num_heads=Hq, decay_factor=0.9, carry_scores=True)
    m_fn, m_slab = H2OScoreSlab(**args), H2OScoreSlab(**args)
    k0, v0 = _rows(gen, L, B, Hkv, D, BUDGET - 5, 0, dt)
    kv = [(k0[l], v0[l]) for l in range(L)]
    slab = KVSlabCache.from_legacy_cache(kv, capacity=BUDGET + 8)
    ref = [None] * L
    t = BUDGET - 5
    compressions = 0
    for step in range(50):
        kn, vn = _rows(gen, L, B, Hkv, D, 1, t, dt)
        t += 1
        kv = [(torch.cat([kv[l][0], kn[l]], 2), torch.cat([kv[l][1], vn[l]], 2)) for l in range(L)]
        slab.append([(kn[l], vn[l]) for l in range(L)])
        S = kv[0][0].size(2)
        attn = [torch.softmax(3 * torch.randn(B, Hq, 1, S, generator=gen, device="cuda"), -1).to(dt) for _ in range(L)]
        for l in range(L):
            prev = ref[l]
            base = torch.zeros(B, Hq, S, dtype=dt, device="cuda")
            if prev is not None:
                base[..., :prev.size(-1)] = prev * 0.9
            ref[l] = base + attn[l].sum(2)
        m_fn.update_attention_scores(attn)
        m_slab.update_attention_scores(attn)
        for l in range(L):
            assert torch.equal(m_fn.accumulated_attention[l], ref[l]), (step, l)
        if S <= BUDGET:
            continue
        compressions += 1
        lo, hi = KW["start_size"], S - KW["recent_size"]
        scores = [_head_sum(ref[l], lo, hi) for l in range(L)]
        kv = kvcompress.h2o_attention_compress(kv, h2o_manager=m_fn, **KW)
        _, idx = slab.compress_("h2o_attention", h2o_manager=m_slab, return_indices=True, **KW)
        for l in range(L):
            kept = idx[l]                                     # [B, Hkv, C] source rows of the slab path
            for b in range(B):
                for h in range(1, Hkv):
                    assert torch.equal(kept[b, 0], kept[b, h])
                _check_topk(scores[l][b], kept[b, 0, 4:-40].long() - 4, KW["heavy_hitter_size"])
            ref[l] = ref[l].gather(-1, kept.long().repeat_interleave(G, dim=1))
            assert torch.equal(m_fn.accumulated_attention[l], ref[l]), (step, l)
            assert torch.equal(m_slab.accumulated_attention[l], ref[l]), (step, l)
            assert torch.equal(slab[l][0], kv[l][0]) and torch.equal(slab[l][1], kv[l][1])
    assert compressions >= 40 and slab.lengths == [BUDGET] * L


@pytest.mark.parametrize("dtype", ["f32", "bf16"])
def test_cumulative_loop_from_queries(dtype):
    """The same loop through update_from_queries: each update within assert_close_ulp of the torch update of the
    device's previous state; each compaction an exact gather of the device's accumulators; both paths identical."""
    dt = DT[dtype]
    L, B, Hkv, G, D = 2, 2, 2, 4, 64
    Hq = Hkv * G
    gen = torch.Generator(device="cuda").manual_seed(7)
    args = dict(KW, num_layers=L, num_heads=Hq, decay_factor=0.9, carry_scores=True)
    m_fn, m_slab = H2OScoreSlab(**args), H2OScoreSlab(**args)
    k0, v0 = _rows(gen, L, B, Hkv, D, BUDGET - 3, 0, dt)
    kv = [(k0[l], v0[l]) for l in range(L)]
    slab = KVSlabCache.from_legacy_cache(kv, capacity=BUDGET + 8)
    t = BUDGET - 3
    for step in range(45):
        kn, vn = _rows(gen, L, B, Hkv, D, 1, t, dt)
        t += 1
        kv = [(torch.cat([kv[l][0], kn[l]], 2), torch.cat([kv[l][1], vn[l]], 2)) for l in range(L)]
        slab.append([(kn[l], vn[l]) for l in range(L)])
        S = kv[0][0].size(2)
        q = [(2 * torch.randn(B, Hq, 1, D, generator=gen, device="cuda")).to(dt) for _ in range(L)]
        before = [m_fn.accumulated_attention[l].clone() if l in m_fn.accumulated_attention else None
                  for l in range(L)]
        m_fn.update_from_queries(q, [kv[l][0] for l in range(L)])
        m_slab.update_from_queries(q, [slab[l][0] for l in range(L)])
        for l in range(L):
            want = torch.zeros(B, Hq, S, dtype=dt, device="cuda")
            if before[l] is not None:
                want[..., :before[l].size(-1)] = before[l] * 0.9
            want = want + ref_probs(q[l], kv[l][0]).sum(2)
            assert_close_ulp(m_fn.accumulated_attention[l], want, f"step {step} layer {l}")
            assert torch.equal(m_fn.accumulated_attention[l], m_slab.accumulated_attention[l])
        if S <= BUDGET:
            continue
        acc = [m_fn.accumulated_attention[l].clone() for l in range(L)]
        kv = kvcompress.h2o_attention_compress(kv, h2o_manager=m_fn, **KW)
        _, idx = slab.compress_("h2o_attention", h2o_manager=m_slab, return_indices=True, **KW)
        for l in range(L):
            want = acc[l].gather(-1, idx[l].long().repeat_interleave(G, dim=1))
            assert torch.equal(m_fn.accumulated_attention[l], want) and torch.equal(m_slab.accumulated_attention[l], want)
            assert torch.equal(slab[l][0], kv[l][0]) and torch.equal(slab[l][1], kv[l][1])


# ---------------------------------------------------------------------------------------------- 3. harness
def torch_cumulative_h2o(model, ids, start_size, heavy_hitter_size, recent_size, decay=0.9):
    """Pure-torch cumulative H2O (eager attention, DynamicCache, fp32): update once per forward, keep sinks + top-k of
    the head-summed accumulators + recent rows, gather the accumulators with the kept rows, never reset."""
    from transformers import DynamicCache

    budget = start_size + heavy_hitter_size + recent_size
    cache, acc, nlls = DynamicCache(), {}, []
    with torch.inference_mode():
        for idx in range(ids.size(1) - 1):
            out = model(ids[:, idx:idx + 1], past_key_values=cache, use_cache=True, output_attentions=True)
            logits = out.logits[:, -1, :].float()
            nlls.append(float(torch.nn.functional.cross_entropy(logits, ids[:, idx + 1]).item()))
            for l, attn in enumerate(out.attentions):
                S = attn.size(-1)
                base = torch.zeros(attn.shape[0], attn.shape[1], S, dtype=attn.dtype, device=attn.device)
                if l in acc:
                    base[..., :acc[l].size(-1)] = acc[l] * decay
                acc[l] = base + attn.sum(2)
            cache = out.past_key_values
            kv = list(normalize_kv_cache(cache))
            S = kv[0][0].size(2)
            if S <= budget:
                continue
            new = []
            for l, (k, v) in enumerate(kv):
                lo, hi = start_size, S - recent_size
                score = acc[l][:, :, lo:hi].sum(1)[0]
                top = torch.sort(torch.topk(score, min(heavy_hitter_size, hi - lo)).indices).values + lo
                kept = torch.cat([torch.arange(start_size, device=k.device), top,
                                  torch.arange(S - recent_size, S, device=k.device)])
                new.append((k[:, :, kept], v[:, :, kept]))
                acc[l] = acc[l][:, :, kept]
            cache = to_dynamic_cache(new)
    return nlls


@pytest.mark.parametrize("cache", ["dynamic", "slab"])
def test_harness_cumulative_matches_a_torch_loop(cache):
    """evaluate_with_attention_compression(carry_scores=True) with scores="attentions" and scores="queries": the
    golden case's cache lengths, per-token NLLs within 5e-3 of the pure-torch cumulative loop."""
    import harness_cases as H
    from kvcompress.evaluate_attention import evaluate_with_attention_compression

    golden = json.load(open(os.path.join(GOLDEN_DIR, "harness_golden.json")))
    want_lengths = golden["cases"]["h2o_attention"]["lengths"]
    model, ids = H.tiny_model_and_ids("cuda", attn_implementation="eager")
    ids = ids.cuda()
    ref = torch_cumulative_h2o(model, ids, **H.ATTN_KW)
    for scores in ("attentions", "queries"):
        n0 = _engine.launch_count()
        got = evaluate_with_attention_compression(model, input_ids=ids, skip_layers=[], show_progress=False,
                                                  return_nlls=True, cache=cache, scores=scores, carry_scores=True,
                                                  **H.ATTN_KW)
        assert _engine.launch_count() > n0
        assert got["cache_lengths"] == want_lengths, scores
        assert got["num_tokens"] == H.TOKENS - 1
        worst = max(abs(a - b) for a, b in zip(got["nlls"], ref))
        assert worst < 5e-3, (scores, worst)


# ---------------------------------------------------------------------------------------------- 4. hot path
def test_one_cumulative_decode_step_is_three_launches_without_aten_or_sync():
    """update_from_queries + compress_ on a slab with carry_scores=True at steady state: stats, accumulate and the
    compaction (which carries the accumulators) — three launches, no ATen kernel, no synchronising call."""
    L, B, Hq, Hkv, D = 4, 2, 8, 2, 64
    gen = torch.Generator(device="cuda").manual_seed(6)
    k, v = torch.randn(B, Hkv, BUDGET + 1, D, generator=gen, device="cuda").bfloat16(), \
        torch.randn(B, Hkv, BUDGET + 1, D, generator=gen, device="cuda").bfloat16()
    slab = KVSlabCache.from_legacy_cache([(k, v)] * L, capacity=BUDGET + 8)
    dev = H2OScoreSlab(num_layers=L, num_heads=Hq, carry_scores=True, **KW)
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
    assert slab.lengths == [BUDGET] * L
    assert all(dev._lens[l] == BUDGET for l in range(L))
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert names and all("kvc_" in n for n in names), names
    assert sum("kvc_h2o_qk_stats_kernel" in n for n in names) == 1
    assert sum("kvc_h2o_qk_accumulate_kernel" in n for n in names) == 1
    assert sum("kvc_slab_compress_kernel" in n for n in names) == 1
