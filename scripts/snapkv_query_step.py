"""SnapKV votes from the model's own queries (SnapKVQueryWindow + the tcgen05 vote) on the GPU, bf16.

  decode    at a Pythia-2.8B shape (32 layers, 32 heads, D 80, G 1, B 1, keep 512) and a Llama-3-8B GQA shape (32 layers,
            Hkv 8, G 4, D 128, B 8, keep 1024), W 32, a cache of keep + 1 rows and a full window, per call:
              push      SnapKVQueryWindow.push of one decode query per head (kvc_query_window_push, one launch);
              vote      the vote alone over the slab's keys (kvc_snapkv_vote), the middle launch of the slab step;
              slab      push + compress_("snapkv_lite", obs_queries=window): push, vote, in-place compaction;
              function  push + snapkv_lite_compress(kv, obs_queries=window): push, fused vote-compress;
              norms     compress_("snapkv_lite") without queries (the norm-based step, one launch);
              h2o       H2OScoreSlab.update_from_queries + compress_("h2o_attention") (the H2O query step, 4/64/rest).
            CUDA events around each call, medians of alternating rounds; the slab is re-grown by one row between calls
            outside the timed region.  The cache (0.7 GB / 2.1 GB of K and V with the Llama shape) is partly
            L2-resident between calls at the Pythia shape (168 MB of K and V over 126 MB of L2).
  prefill   a 4096-token prompt compressed to 1024 at both shapes: push of T = 4096 from an empty window plus the fused
            vote-compress (function path).

    python scripts/snapkv_query_step.py --out profiles/r07_snapkv_query_step.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs3602-llm-inference-acceleration_b200"))
import torch  # noqa: E402

import kvcompress  # noqa: E402
from kvcompress import H2OScoreSlab, KVSlabCache, QueryCapture, SnapKVQueryWindow, _engine  # noqa: E402

SHAPES = {
    # name: L, B, Hq, Hkv, D, keep
    "pythia2.8b_b1_keep512": (32, 1, 32, 32, 80, 512),
    "llama3_8b_gqa_b8_keep1024": (32, 8, 32, 8, 128, 1024),
}
W = 32


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def timed(fn, reps, between=None):
    """Median ms per call from CUDA events around each call; `between` runs untimed after each call."""
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        if between is not None:
            between()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    out.sort()
    return out[len(out) // 2]


def hf_queries(B, Hq, T, D, g):
    return (1.5 * torch.randn(B, T, Hq, D, generator=g, device="cuda")).bfloat16().transpose(1, 2)


def capture(qs, keys):
    cap = QueryCapture(len(qs))
    for l, q in enumerate(qs):
        cap._record(l, q, keys[l], None, q.size(-1) ** -0.5)
    return cap


def decode(name, rounds, reps):
    L, B, Hq, Hkv, D, keep = SHAPES[name]
    g = torch.Generator(device="cuda").manual_seed(0)
    S = keep + 1
    kv = [(torch.randn(B, Hkv, S, D, generator=g, device="cuda").bfloat16(),
           torch.randn(B, Hkv, S, D, generator=g, device="cuda").bfloat16()) for _ in range(L)]
    new = [(k[:, :, :1].contiguous(), v[:, :, :1].contiguous()) for k, v in kv]
    slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
    win = SnapKVQueryWindow(L, B, Hq, D, W, torch.bfloat16, "cuda")
    win.push([hf_queries(B, Hq, W, D, g) for _ in range(L)])
    qs = [hf_queries(B, Hq, 1, D, g) for _ in range(L)]
    cap = capture(qs, [slab[l][0] for l in range(L)])
    kw = dict(observation_window=W, keep_size=keep, skip_layers=[])
    heavy = 64
    h2o_kw = dict(start_size=4, heavy_hitter_size=heavy, recent_size=keep - 4 - heavy)
    h2o = H2OScoreSlab(num_layers=L, num_heads=Hq, **h2o_kw)
    regrow = lambda: slab.append(new)  # noqa: E731

    def h2o_step():
        h2o.update_from_queries(cap.queries, cap.keys, cap.masks, cap.scaling)
        slab.compress_("h2o_attention", h2o_manager=h2o, **h2o_kw)
        h2o.reset()

    paths = {
        "push": (lambda: win.push(cap), None),
        "vote": (lambda: _engine.snapkv_votes([(slab[l][0], win.queries[l]) for l in range(L)], W), None),
        "slab": (lambda: (win.push(cap), slab.compress_("snapkv_lite", obs_queries=win, **kw)), regrow),
        "function": (lambda: (win.push(cap), kvcompress.snapkv_lite_compress(kv, obs_queries=win, **kw)), None),
        "norms": (lambda: slab.compress_("snapkv_lite", **kw), regrow),
        "h2o": (h2o_step, regrow),
    }
    launches = {}
    for k, (fn, between) in paths.items():
        for _ in range(3):
            fn()
            if between:
                between()
        torch.cuda.synchronize()
        n0 = _engine.launch_count()
        fn()
        launches[k] = _engine.launch_count() - n0
        if between:
            between()
    med = {k: [] for k in paths}
    for _ in range(rounds):
        for k, (fn, between) in paths.items():
            med[k].append(timed(fn, reps, between))
    res = {k: sorted(v)[len(v) // 2] for k, v in med.items()}
    # per-kernel split of the slab step from the profiler, in a run of its own
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        paths["slab"][0]()
        torch.cuda.synchronize()
    regrow()
    kernels = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            key = ev.name.split("<")[0].split("(")[0][:60]
            kernels[key] = round(kernels.get(key, 0.0) + ev.device_time_total, 2)
    e = 2
    return {"shape": dict(zip(("L", "B", "Hq", "Hkv", "D", "keep"), SHAPES[name]), W=W, S=S), "dtype": "bf16",
            "K_bytes": L * B * Hkv * S * D * e, "window_bytes": L * B * Hq * W * D * e,
            "launches": launches, "ms_median": res, "ms_per_round": med, "slab_step_profiler_us": kernels,
            "vote_share_of_slab_step": res["vote"] / res["slab"]}


def prefill(name, reps, T=4096, keep=1024):
    L, B, Hq, Hkv, D, _ = SHAPES[name]
    g = torch.Generator(device="cuda").manual_seed(1)
    kv = [(torch.randn(B, Hkv, T, D, generator=g, device="cuda").bfloat16(),
           torch.randn(B, Hkv, T, D, generator=g, device="cuda").bfloat16()) for _ in range(L)]
    qs = [hf_queries(B, Hq, T, D, g) for _ in range(L)]
    win = SnapKVQueryWindow(L, B, Hq, D, W, torch.bfloat16, "cuda")
    kw = dict(observation_window=W, keep_size=keep, skip_layers=[])

    def push():
        win.reset()
        win.push(qs)

    def step():
        push()
        kvcompress.snapkv_lite_compress(kv, obs_queries=win, **kw)

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    return {"shape": dict(zip(("L", "B", "Hq", "Hkv", "D"), SHAPES[name][:5]), T=T, keep=keep, W=W),
            "K_bytes": L * B * Hkv * T * D * 2, "push_ms_median": timed(push, reps),
            "push_plus_vote_compress_ms_median": timed(step, reps)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07_snapkv_query_step.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    res = {"gpu": gpu_info(), "method": "CUDA events per call, median over reps, median of alternating rounds",
           "decode": {n: decode(n, args.rounds, args.reps) for n in SHAPES},
           "prefill": {n: prefill(n, 10) for n in SHAPES}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({n: r["ms_median"] for n, r in res["decode"].items()}, indent=1))
    print(json.dumps(res["prefill"], indent=1))


if __name__ == "__main__":
    main()
