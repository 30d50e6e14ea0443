"""-m gpu: SnapKV votes from the model's own queries — SnapKVQueryWindow (kvc_query_window_push) against torch slicing,
the vote fed from the window against the same vote from torch-built queries and an fp64 torch SnapKV step, lockstep
decode on tiny bf16 HF models through the function and the slab path, the harnesses with scores="queries", and the
launches of a steady decode step."""

import pytest
import torch
from torch.utils._python_dispatch import TorchDispatchMode

import kvcompress
from kvcompress import KVSlabCache, QueryCapture, SnapKVQueryWindow, _engine, _planner
from kvcompress.benchmark import measure_generation_metrics
from kvcompress.evaluate import evaluate_with_compression, new_slab_for_model
from kvcompress.utils import normalize_kv_cache, to_dynamic_cache

pytestmark = pytest.mark.gpu

ULP = {torch.bfloat16: 2.0 ** -8, torch.float16: 2.0 ** -11}


def hf_queries(B, Hq, T, D, dtype, gen):
    """[B, Hq, T, D] as HF attention hands it over: a transpose of [B, T, Hq, D] (last dim dense, other strides not)."""
    return torch.randn(B, T, Hq, D, generator=gen, device="cuda").to(dtype).transpose(1, 2)


def capture_of(queries):
    cap = QueryCapture(len(queries))
    for l, q in enumerate(queries):
        cap._record(l, q, None, None, q.size(-1) ** -0.5)
    return cap


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("Hq,D", [(2, 64), (8, 80), (16, 128)])   # G 1 / 4 / 8 over Hkv 2
@pytest.mark.parametrize("start_full", [False, True])
def test_push_is_bit_exact_against_torch(dtype, Hq, D, start_full):
    """Sequences of pushes (n_new 1, 7, W-1, W, 3W, per layer in a different order, some layers not run) from filled 0
    or W: the valid rows equal torch's cat-and-slice bit for bit, and every push is exactly one launch."""
    L, B, W = 5, 2, 32
    gen = torch.Generator(device="cuda").manual_seed(Hq + D)
    win = SnapKVQueryWindow(L, B, Hq, D, W, dtype, "cuda")
    ref = [torch.empty(B, Hq, 0, D, dtype=dtype, device="cuda") for _ in range(L)]
    if start_full:
        first = [hf_queries(B, Hq, W, D, dtype, gen) for _ in range(L)]
        win.push(capture_of(first))
        ref = [q.clone() for q in first]
        assert win.filled == [W] * L
    sizes = [1, 7, W - 1, W, 3 * W, 1, 1]
    for step in range(len(sizes)):
        new = [None if (l + step) % 4 == 3 else hf_queries(B, Hq, sizes[(l + step) % len(sizes)], D, dtype, gen)
               for l in range(L)]
        n0 = _engine.launch_count()
        win.push(new)
        assert _engine.launch_count() - n0 == 1
        for l in range(L):
            if new[l] is not None:
                ref[l] = torch.cat([ref[l], new[l]], dim=2)[:, :, -W:]
            assert win.filled[l] == ref[l].size(2)
            assert torch.equal(win.queries[l][:, :, :win.filled[l]], ref[l]), (step, l)


def test_many_layers_one_launch_per_64():
    L, B, Hq, D, W = 70, 1, 4, 64, 16
    gen = torch.Generator(device="cuda").manual_seed(2)
    win = SnapKVQueryWindow(L, B, Hq, D, W, torch.bfloat16, "cuda")
    qs = [hf_queries(B, Hq, 20, D, torch.bfloat16, gen) for _ in range(L)]
    n0 = _engine.launch_count()
    win.push(qs)
    assert _engine.launch_count() - n0 == 2
    for l in range(L):
        assert torch.equal(win.queries[l], qs[l][:, :, -W:])


def ref_votes(keys, queries, window):
    """fp64 SnapKV vote: logits x D^-0.5, causal inside the window, softmax over all keys, sum over window and group."""
    B, H, S, D = keys.shape
    G = queries.size(1) // H
    k = keys.double().repeat_interleave(G, dim=1)
    s = torch.matmul(queries.double(), k.transpose(-1, -2)) * D ** -0.5
    pos_q = (S - window) + torch.arange(window, device=keys.device).view(window, 1)
    s = s.masked_fill(torch.arange(S, device=keys.device).view(1, S) > pos_q, float("-inf"))
    return torch.softmax(s, -1)[..., :S - window].sum(2).view(B, H, G, -1).sum(2)


def pooled(votes, pk=5):
    B, H, P = votes.shape
    return torch.nn.functional.avg_pool1d(votes.reshape(B * H, 1, P), pk, 1, pk // 2).reshape(B, H, P)


def check_choice(ref_pool, idx, k, dtype, what):
    """Kept prefix rows (ascending) are a top-k of the fp64 pooled votes, up to the error of the device's pooled 16-bit
    votes (2.5 ulps per vote, one more rounding, a margin): no kept row is below the k-th score and no dropped row
    above it by more than that."""
    for b in range(ref_pool.size(0)):
        for h in range(ref_pool.size(1)):
            s, rows = ref_pool[b, h], idx[b, h, :k].long()
            assert rows.numel() == k and bool((rows[1:] > rows[:-1]).all()), what
            kth = torch.topk(s, k).values[-1]
            tol = 4 * ULP[dtype] * float(kth) + 1e-7
            kept = torch.zeros_like(s, dtype=torch.bool)
            kept[rows] = True
            assert bool((s[kept] >= kth - tol).all()) and bool((s[~kept] <= kth + tol).all()), (what, b, h)


@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float16])
@pytest.mark.parametrize("B,Hkv,G,D", [(1, 2, 1, 80), (2, 2, 4, 128), (1, 1, 4, 64)])
def test_vote_from_the_window(dtype, B, Hkv, G, D):
    """The window as obs_queries: votes and kept rows bit-identical to the same call with torch-built queries; votes
    within test_gpu_vote's tolerance of fp64; kept rows a tie-aware top-k; K / V a torch gather; the slab path keeps
    the same rows."""
    L, S, W, keep = 3, 300, 32, 96
    gen = torch.Generator(device="cuda").manual_seed(B * 10 + G)
    kv = [(torch.randn(B, Hkv, S, D, generator=gen, device="cuda").to(dtype),
           torch.randn(B, Hkv, S, D, generator=gen, device="cuda").to(dtype)) for _ in range(L)]
    win = SnapKVQueryWindow(L, B, Hkv * G, D, W, dtype, "cuda")
    hist = [torch.empty(B, Hkv * G, 0, D, dtype=dtype, device="cuda") for _ in range(L)]
    for T in (40, 1, 1, 3):   # a prompt, then decode-sized pushes
        qs = [(1.5 * hf_queries(B, Hkv * G, T, D, torch.float32, gen)).to(dtype) for _ in range(L)]
        win.push(qs)
        hist = [torch.cat([h, q], 2)[:, :, -W:] for h, q in zip(hist, qs)]
    plans = [_planner.LayerPlan(_planner.GATHER, S, 0, 0, S - W, keep - W, W, _planner.SCORE_GIVEN_SCORE, 5)] * L
    out_w, idx_w, votes_w = _engine.snapkv_vote_compress(kv, plans, win.queries, W, return_indices=True,
                                                         return_votes=True)
    out_t, idx_t, votes_t = _engine.snapkv_vote_compress(kv, plans, [h.contiguous() for h in hist], W,
                                                         return_indices=True, return_votes=True)
    fn = kvcompress.snapkv_lite_compress(kv, observation_window=W, keep_size=keep, obs_queries=win, skip_layers=[])
    slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
    slab.compress_("snapkv_lite", observation_window=W, keep_size=keep, obs_queries=win, skip_layers=[])
    for l in range(L):
        assert torch.equal(votes_w[l], votes_t[l]) and torch.equal(idx_w[l], idx_t[l])
        assert torch.equal(out_w[l][0], out_t[l][0]) and torch.equal(out_w[l][1], out_t[l][1])
        want = ref_votes(kv[l][0], hist[l], W)
        got = votes_w[l].double()
        assert torch.all((got - want).abs() <= 2.5 * ULP[dtype] * want + 1e-7), l
        check_choice(pooled(want), idx_w[l], keep - W, dtype, f"layer {l}")
        rows = idx_w[l].long().unsqueeze(-1).expand(-1, -1, -1, D)
        assert torch.equal(out_w[l][0], torch.gather(kv[l][0], 2, rows))
        assert torch.equal(out_w[l][1], torch.gather(kv[l][1], 2, rows))
        assert torch.equal(fn[l][0], out_w[l][0]) and torch.equal(fn[l][1], out_w[l][1])
        assert torch.equal(slab[l][0], out_w[l][0]) and torch.equal(slab[l][1], out_w[l][1])


def _tiny(kind):
    """Tiny bf16 models with head dims the vote covers: GPT-NeoX MHA (D 64, G 1) and Llama GQA (D 64, G 4)."""
    from transformers import GPTNeoXConfig, GPTNeoXForCausalLM, LlamaConfig, LlamaForCausalLM

    torch.manual_seed(0)
    if kind == "neox":
        cfg = GPTNeoXConfig(vocab_size=256, hidden_size=256, num_hidden_layers=3, num_attention_heads=4,
                            intermediate_size=256, max_position_embeddings=512, rotary_pct=0.25)
        return GPTNeoXForCausalLM(cfg).eval().cuda().bfloat16()
    cfg = LlamaConfig(vocab_size=256, hidden_size=512, num_hidden_layers=3, num_attention_heads=8,
                      num_key_value_heads=2, intermediate_size=256, max_position_embeddings=512)
    return LlamaForCausalLM(cfg).eval().cuda().bfloat16()


@pytest.mark.parametrize("kind", ["neox", "llama_gqa"])
def test_lockstep_decode_on_tiny_models(kind):
    """A prompt, then 50 decode steps (40+ past the budget) on a slab: at every compressing step the window equals the
    torch window of the captured queries, the device's choice is valid against fp64 SnapKV on the same cache, and the
    function path keeps exactly the slab path's rows."""
    model = _tiny(kind)
    cfg = model.config
    L, W, keep, B = cfg.num_hidden_layers, 8, 32, 2
    ids = torch.randint(0, cfg.vocab_size, (B, 24 + 50), generator=torch.Generator().manual_seed(3)).cuda()
    slab = new_slab_for_model(model, B, capacity=128)
    cache = slab.as_hf_cache()
    win = SnapKVQueryWindow.for_model(model, B, W)
    hist = [None] * L
    kw = dict(observation_window=W, keep_size=keep, skip_layers=[])
    compressed = 0
    with torch.inference_mode():
        for a, b in [(0, 24)] + [(p, p + 1) for p in range(24, 74)]:
            with kvcompress.capture_queries(model) as cap:
                model(ids[:, a:b], past_key_values=cache, use_cache=True)
            assert all(m is None for m in cap.masks)
            win.push(cap)
            hist = [cap.queries[l] if h is None else torch.cat([h, cap.queries[l]], 2)[:, :, -W:]
                    for l, h in enumerate(hist)]
            if slab.lengths[0] <= keep:
                continue
            compressed += 1
            kv = [(k.clone(), v.clone()) for k, v in slab]
            for l in range(L):
                assert torch.equal(win.queries[l], hist[l])
            fn = kvcompress.snapkv_lite_compress(kv, obs_queries=win, **kw)
            _, idx = slab.compress_("snapkv_lite", return_indices=True, obs_queries=win, **kw)
            for l in range(L):
                assert torch.equal(slab[l][0], fn[l][0]) and torch.equal(slab[l][1], fn[l][1]), (a, l)
                check_choice(pooled(ref_votes(kv[l][0], hist[l], W)), idx[l], keep - W, torch.bfloat16, (a, l))
            assert slab.lengths == [keep] * L
    assert compressed >= 40 and win.num_heads == cfg.num_attention_heads


def torch_snapkv_nlls(model, ids, W, keep, skip):
    """The pure-torch loop: DynamicCache, a torch window of captured queries, fp64 votes, avg_pool1d, top-k, sort,
    gather, one token per forward, NLLs computed as the harness computes them."""
    from transformers import DynamicCache

    L = model.config.num_hidden_layers
    cache, hist, nlls = DynamicCache(), [None] * L, []
    loss = torch.nn.CrossEntropyLoss(reduction="none")
    with torch.inference_mode():
        for i in range(ids.size(1) - 1):
            with kvcompress.capture_queries(model) as cap:
                out = model(ids[:, i:i + 1], past_key_values=cache, use_cache=True)
            hist = [q if h is None else torch.cat([h, q], 2)[:, :, -W:] for h, q in zip(hist, cap.queries)]
            logits = out.logits[:, -1, :].view(-1, model.config.vocab_size)   # as the harness computes it
            nlls.append(float(loss(logits, ids[:, i + 1:i + 2].view(-1)).mean()))
            kv = list(normalize_kv_cache(out.past_key_values))
            new = []
            for l, (k, v) in enumerate(kv):
                S = k.size(2)
                if l in skip or S <= keep:
                    new.append((k, v))
                    continue
                # the device's rounding points: votes and pooled votes in the cache dtype; ties to the lowest row
                votes = ref_votes(k, hist[l], W).to(k.dtype).float()
                score = pooled(votes).to(k.dtype)
                top = torch.sort(score, dim=-1, descending=True, stable=True).indices[..., :keep - W].sort(-1).values
                rows = torch.cat([top, torch.arange(S - W, S, device=k.device).expand(*top.shape[:2], W)], -1)
                g = rows.unsqueeze(-1).expand(-1, -1, -1, k.size(3))
                new.append((torch.gather(k, 2, g), torch.gather(v, 2, g)))
            cache = to_dynamic_cache(new)
    return nlls


@pytest.mark.parametrize("cache", ["dynamic", "slab"])
def test_evaluate_with_queries_matches_a_torch_snapkv_loop(cache):
    import harness_cases as H

    model, ids = H.tiny_model_and_ids("cuda")
    model = model.bfloat16()
    ids = ids.cuda()
    kw = dict(observation_window=8, keep_size=32, pooling_kernel=5)
    got = evaluate_with_compression(model, input_ids=ids, compress_fn=kvcompress.snapkv_lite_compress,
                                    compress_kwargs=kw, skip_layers=H.SKIP, show_progress=False, return_nlls=True,
                                    cache=cache, scores="queries")
    S = H.TOKENS - 1
    assert got["cache_lengths"] == [S if l in H.SKIP else 32 for l in range(model.config.num_hidden_layers)]
    assert got["final_cache_size"] == 32 and got["num_tokens"] == S
    want = torch_snapkv_nlls(model, ids, 8, 32, H.SKIP)
    # the NLLs of a bf16 model are bf16 (one ulp is 2^-5 at 4..8): a near-tie vote the device and fp64 round apart can
    # keep another row and move a later token's NLL by an ulp or two, so the mean is held to 5e-3 and each token to
    # four ulps
    diff = [abs(a - b) for a, b in zip(got["nlls"], want)]
    assert sum(diff) / len(diff) < 5e-3 and max(diff) <= 0.125, (sum(diff) / len(diff), max(diff))


def test_norms_results_are_unchanged():
    import harness_cases as H

    model, ids = H.tiny_model_and_ids("cuda")
    model = model.bfloat16()
    kw = dict(observation_window=8, keep_size=32, pooling_kernel=5)
    args = dict(input_ids=ids.cuda(), compress_fn=kvcompress.snapkv_lite_compress, compress_kwargs=kw,
                skip_layers=H.SKIP, show_progress=False, return_nlls=True, cache="slab")
    a = evaluate_with_compression(model, **args)
    b = evaluate_with_compression(model, scores="norms", **args)
    assert a["nlls"] == b["nlls"] and a["cache_lengths"] == b["cache_lengths"]


@pytest.mark.parametrize("cache", ["dynamic", "slab"])
def test_generation_with_queries(cache):
    model = _tiny("llama_gqa")
    ids = torch.randint(0, 256, (2, 40), generator=torch.Generator().manual_seed(4)).cuda()
    res = measure_generation_metrics(model, input_ids=ids, compress_fn=kvcompress.snapkv_lite_compress,
                                     compress_kwargs=dict(observation_window=8, keep_size=32), max_new_tokens=24,
                                     skip_layers=[0], cache=cache, scores="queries")
    assert res["num_tokens"] == 24 and res["input_length"] == 40


class AtenOps(TorchDispatchMode):
    """Every ATen op dispatched inside the context.  A step that dispatches only views, empty allocations and
    metadata queries cannot have launched an ATen kernel."""

    def __init__(self):
        super().__init__()
        self.ops = []

    def __torch_dispatch__(self, func, types, args=(), kwargs=None):
        self.ops.append(func)
        return func(*args, **(kwargs or {}))

    def kernel_ops(self):
        return [str(op) for op in self.ops
                if not (op.is_view or op.overloadpacket in (torch.ops.aten.empty, torch.ops.aten.empty_strided,
                                                            torch.ops.aten.is_pinned))]


def test_steady_step_launches_without_aten_or_sync():
    """At steady state: slab = push + vote + in-place compaction (3 library launches), function path = push + fused
    vote-compress (2); no ATen op that launches a kernel, no synchronising call."""
    L, B, Hkv, G, D, W, keep = 4, 2, 2, 4, 64, 16, 64
    gen = torch.Generator(device="cuda").manual_seed(6)
    k, v = (torch.randn(B, Hkv, keep + 1, D, generator=gen, device="cuda").bfloat16() for _ in range(2))
    slab = KVSlabCache.from_legacy_cache([(k, v)] * L, capacity=keep + 8)
    win = SnapKVQueryWindow(L, B, Hkv * G, D, W, torch.bfloat16, "cuda")
    win.push([hf_queries(B, Hkv * G, W, D, torch.bfloat16, gen) for _ in range(L)])
    cap = capture_of([hf_queries(B, Hkv * G, 1, D, torch.bfloat16, gen) for _ in range(L)])
    kw = dict(observation_window=W, keep_size=keep, skip_layers=[])
    kv = [(k, v)] * L
    new = [(k[:, :, :1].contiguous(), v[:, :, :1].contiguous())] * L

    def slab_step():
        win.push(cap)
        slab.compress_("snapkv_lite", obs_queries=win, **kw)

    def fn_step():
        win.push(cap)
        kvcompress.snapkv_lite_compress(kv, obs_queries=win, **kw)

    for step, launches in ((slab_step, 3), (fn_step, 2)):
        step()                  # warm-up: plan caches
        if step is slab_step:
            slab.append(new)    # back to keep + 1 rows
        torch.cuda.synchronize()
        n0 = _engine.launch_count()
        torch.cuda.set_sync_debug_mode("error")
        try:
            with AtenOps() as aten:
                step()
        finally:
            torch.cuda.set_sync_debug_mode(0)
        torch.cuda.synchronize()
        assert _engine.launch_count() - n0 == launches
        assert aten.kernel_ops() == [], aten.kernel_ops()
    assert slab.lengths == [keep] * L
