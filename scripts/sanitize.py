#!/usr/bin/env python
"""Small-shape exerciser for compute-sanitizer (memcheck / racecheck / synccheck / initcheck) over every kernel
family of the library: the fused kernel (scan, stored norms, caller rows, caller scores, workspace, generic row
width), slab append (both forms), in-place compaction (overlapping source / destination), the tcgen05 vote (two
passes, single pass, fused tail), the tensor-core H2O query update (both passes, causal and masked tiles), the SnapKV observation-window push.  Results
are checked against torch (or the CUDA-core form) so a sanitizer-clean run is also a correct one.

    compute-sanitizer --tool racecheck python scripts/sanitize.py
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import lab_util  # noqa: E402,F401

import torch  # noqa: E402

import kvcompress  # noqa: E402
from kvcompress import KVSlabCache, _engine, _planner  # noqa: E402


def rows(B, H, T, D, dt, gen):
    k = torch.randn(B, H, T, D, generator=gen, device="cuda") * torch.exp(0.35 * torch.randn(B, H, T, 1, generator=gen, device="cuda"))
    return k.to(dt), torch.randn(B, H, T, D, generator=gen, device="cuda").to(dt)


def main():
    gen = torch.Generator(device="cuda").manual_seed(1)
    n0 = _engine.launch_count()
    for dt, D in ((torch.bfloat16, 80), (torch.float32, 128), (torch.float16, 72)):
        L, B, H, S = 2, 2, 2, 700
        kv = [rows(B, H, S, D, dt, gen) for _ in range(L)]
        ref = kvcompress.h2o_l2_compress(kv, start_size=4, heavy_hitter_size=32, recent_size=92)          # scan
        kvcompress.streaming_llm_compress(kv, start_size=4, recent_size=124)                             # pure slice
        kvcompress.snapkv_lite_compress(kv, observation_window=16, keep_size=128)                        # pooling transform
        kvcompress.fix_size_l2_compress(kv, fix_kv_size=128, keep_ratio=0.25, strategy="random", skip_layers=[])  # caller rows
        slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 4)                                          # bulk-copy append
        by_norms = kvcompress.h2o_l2_compress(slab, start_size=4, heavy_hitter_size=32, recent_size=92)  # stored norms
        slab.compress_("h2o_l2", start_size=4, heavy_hitter_size=32, recent_size=92)                     # in place
        for li in range(L):
            assert torch.equal(by_norms[li][0], ref[li][0]) and torch.equal(slab[li][0], ref[li][0])
            assert torch.equal(by_norms[li][1], ref[li][1]) and torch.equal(slab[li][1], ref[li][1])
        new = [rows(B, H, 1, D, dt, gen) for _ in range(L)]
        slab.append(new)                                                                                 # row-per-thread append
        slab.update(new[0][0], new[0][1], 0)                                                             # one-layer append
        slab.compress_("streaming_llm", start_size=4, recent_size=100)                                    # in-place memmove
    # selection beyond shared memory: keys / kept rows in the device workspace
    big = [rows(1, 2, 70000, 16, torch.float32, gen)]
    kvcompress.l2_compress(big, keep_ratio=0.5, prune_after=100, skip_layers=[])
    # the vote: two passes, single pass (caller LSE), fused tail
    for (B, H, G, W, S, D, dt) in ((1, 2, 4, 32, 700, 128, torch.bfloat16), (2, 2, 1, 32, 500, 80, torch.bfloat16),
                                   (1, 2, 2, 16, 300, 64, torch.float16)):
        k, v = rows(B, H, S, D, dt, gen)
        q = (1.5 * torch.randn(B, H * G, W, D, generator=gen, device="cuda")).to(dt)
        kf = k.float().repeat_interleave(G, dim=1)
        sc = torch.matmul(q.float(), kf.transpose(-1, -2)) / D ** 0.5
        pos_q = (S - W) + torch.arange(W, device="cuda").view(1, 1, W, 1)
        sc = sc.masked_fill(torch.arange(S, device="cuda").view(1, 1, 1, S) > pos_q, float("-inf"))
        want = torch.softmax(sc, -1)[..., :S - W].sum(2).view(B, H, G, -1).sum(2)
        lse = torch.logsumexp(sc, -1)
        ulp = 2.0 ** -8 if dt == torch.bfloat16 else 2.0 ** -11
        for votes in (_engine.snapkv_votes([(k, q)], W)[0], _engine.snapkv_votes([(k, q)], W, lse=[lse])[0]):
            assert torch.all((votes.float() - want).abs() <= 2.5 * ulp * want + 1e-7)
        plan = [_planner.LayerPlan(_planner.GATHER, S, 0, 0, S - W, 96 - W, W, _planner.SCORE_GIVEN_SCORE, 5)]
        out, idx = _engine.snapkv_vote_compress([(k, v)], plan, [q], W, return_indices=True)
        gathered = torch.gather(v, 2, idx[0].long().unsqueeze(-1).expand(-1, -1, -1, D))
        assert torch.equal(out[0][1], gathered)
    # the tensor-core H2O query update: both passes (causal and masked tiles, D = 80 tail boxes, GQA) + the score row,
    # against the CUDA-core form
    from kvcompress import H2OScoreSlab
    for (B, Hkv, G, T, S, D, dt) in ((1, 2, 4, 40, 300, 128, torch.bfloat16), (2, 1, 1, 130, 200, 80, torch.float16),
                                     (1, 2, 8, 1, 150, 64, torch.bfloat16)):
        q = (2 * torch.randn(B, Hkv * G, T, D, generator=gen, device="cuda")).to(dt)
        k = torch.randn(B, Hkv, S, D, generator=gen, device="cuda").to(dt)
        mask = torch.rand(B, T, S, generator=gen, device="cuda") > 0.3
        for m in (None, mask):
            kw = dict(start_size=4, heavy_hitter_size=16, recent_size=40, num_layers=1, num_heads=Hkv * G)
            tc, cc = H2OScoreSlab(tensor_cores=True, **kw), H2OScoreSlab(**kw)
            tc.update_from_queries([q], [k], masks=[m])
            cc.update_from_queries([q], [k], masks=[m])
            a, b = tc.accumulated_attention[0].double(), cc.accumulated_attention[0].double()
            assert torch.all((a - b).abs() <= 2.0 ** -5 * a.abs().maximum(b.abs()) + 1e-6)
    # the observation-window push: a prompt longer than the window, a decode push that slides every row, a partial
    # window, an HF-strided view, and a row wider than one 256-byte round
    from kvcompress import SnapKVQueryWindow
    for (B, Hq, D, W, dt) in ((2, 4, 80, 32, torch.bfloat16), (1, 2, 256, 8, torch.float16)):
        win = SnapKVQueryWindow(2, B, Hq, D, W, dt, "cuda")
        ref = [torch.empty(B, Hq, 0, D, dtype=dt, device="cuda") for _ in range(2)]
        for T in (5, 3 * W, 1, W - 1):
            qs = [torch.randn(B, T, Hq, D, generator=gen, device="cuda").to(dt).transpose(1, 2) for _ in range(2)]
            win.push(qs)
            ref = [torch.cat([r, q], 2)[:, :, -W:] for r, q in zip(ref, qs)]
            for l in range(2):
                assert torch.equal(win.queries[l][:, :, :win.filled[l]], ref[l])
    torch.cuda.synchronize()
    print(f"sanitize.py ok: {_engine.launch_count() - n0} launches")


if __name__ == "__main__":
    main()
