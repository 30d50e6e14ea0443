"""H2O attention mass from the queries (H2OScoreSlab.update_from_queries, kvc_h2o_accumulate_qk) on the GPU.

  update    the update alone (two launches: stats + accumulate) at the scripts/h2o_step.py decode shapes and at a
            Llama-3-8B GQA shape with B 1 and key_len 32K; CUDA-event time per update, the algorithmic bytes (K read
            twice, q, acc read and written, the score row) over the data-sheet 7.7 TB/s; beside it
            update_attention_scores on same-shaped bf16 attention rows.  Layers x K exceed the 126 MB L2 at 32K; the
            smaller shapes are stated as they are (their K may be partly L2-resident between passes).
  prefill   the update at the Llama GQA shape with T = key_len = 4096 and 16384 (one layer): time and fp32 FLOP/s
            (2 * D multiply-adds per visible (query, key) pair and pass, both passes) against the CUDA-core rate from
            SM count x 128 lanes x 2 x max SM clock; beside it the attentions path at 4096, and the bytes the
            attentions path would need at 16384.
  tpot      the attention-score harness (evaluate_with_attention_compression, cache="slab", H2OScoreSlab, h2o 4/64/444, every layer compressed)
            on a Pythia-2.8B-shaped random-weight bf16 GPT-NeoX at batch 1: eager + output_attentions against
            capture_queries (SDPA), alternating, with the uncompressed per-token forwards of both as context.

    python scripts/h2o_query_step.py --out profiles/r04_h2o_query_step.json
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
from kvcompress import H2OScoreSlab, _engine  # noqa: E402

DATASHEET_TBPS = 7.7
UPDATE_SHAPES = {
    # name: L, B, Hq, Hkv, D, key_len
    "pythia2.8b_b1_s513": (32, 1, 32, 32, 80, 513),
    "llama3_8b_gqa_b8_s1025": (32, 8, 32, 8, 128, 1025),
    "llama3_8b_gqa_b1_s32768": (32, 1, 32, 8, 128, 32768),
}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def events(fn, reps):
    """Median / min ms per call from CUDA events around each call."""
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    out.sort()
    return out[len(out) // 2], out[0]


def manager(L, Hq):
    return H2OScoreSlab(start_size=4, heavy_hitter_size=64, recent_size=444, num_layers=L, num_heads=Hq)


def update_alone(name, rounds, reps):
    L, B, Hq, Hkv, D, S = UPDATE_SHAPES[name]
    dt, e = torch.bfloat16, 2
    g = torch.Generator(device="cuda").manual_seed(0)
    keys = [torch.randn(B, Hkv, S, D, generator=g, device="cuda").to(dt) for _ in range(L)]
    qs = [(2 * torch.randn(B, Hq, 1, D, generator=g, device="cuda")).to(dt) for _ in range(L)]
    attn = [torch.softmax(2 * torch.randn(B, Hq, 1, S, generator=g, device="cuda"), -1).to(dt) for _ in range(L)]
    m_q, m_a = manager(L, Hq), manager(L, Hq)
    paths = {"queries": lambda: m_q.update_from_queries(qs, keys), "attentions": lambda: m_a.update_attention_scores(attn)}
    for fn in paths.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    n0 = _engine.launch_count()
    paths["queries"]()
    launches = _engine.launch_count() - n0
    med = {k: [] for k in paths}
    for _ in range(rounds):   # alternate the two paths
        for k, fn in paths.items():
            med[k].append(events(fn, reps)[0])
    res = {k: sorted(v)[len(v) // 2] for k, v in med.items()}
    region = max(S - 444 - 4, 0)
    bytes_q = L * (2 * B * Hkv * S * D * e + B * Hq * D * e + 2 * B * Hq * S * e + B * region * e)
    bytes_a = L * (B * Hq * S * e + 2 * B * Hq * S * e + B * region * e)
    # a per-pass split from the profiler, in a separate run of its own
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        paths["queries"]()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            key = "stats" if "qk_stats" in ev.name else "accumulate" if "qk_accumulate" in ev.name else ev.name[:60]
            kernels[key] = round(kernels.get(key, 0.0) + ev.device_time_total, 2)
    return {"shape": dict(zip(("L", "B", "Hq", "Hkv", "D", "key_len"), UPDATE_SHAPES[name])), "dtype": "bf16",
            "K_bytes": L * B * Hkv * S * D * e, "launches_per_update": launches,
            "queries_ms_median": res["queries"], "queries_bytes": bytes_q,
            "queries_TBps": bytes_q / res["queries"] / 1e9,
            "queries_fraction_of_datasheet": bytes_q / res["queries"] / 1e9 / DATASHEET_TBPS,
            "profiler_us_per_pass": kernels,
            "attentions_ms_median": res["attentions"], "attentions_bytes": bytes_a,
            "attentions_TBps": bytes_a / res["attentions"] / 1e9}


def prefill(T, reps, with_attentions):
    L, B, Hq, Hkv, D = 1, 1, 32, 8, 128
    dt = torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(1)
    keys = [torch.randn(B, Hkv, T, D, generator=g, device="cuda").to(dt)]
    qs = [(2 * torch.randn(B, Hq, T, D, generator=g, device="cuda")).to(dt)]
    m = manager(L, Hq)
    m.update_from_queries(qs, keys)
    torch.cuda.synchronize()
    med, best = events(lambda: m.update_from_queries(qs, keys), reps)
    visible_pairs = B * Hq * T * (T + 1) // 2
    flop = 2 * 2 * D * visible_pairs   # two passes
    props = torch.cuda.get_device_properties(0)
    clock_mhz = None
    try:
        clock_mhz = float(subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits"],
                                         capture_output=True, text=True, timeout=30).stdout.split()[0])
    except Exception:
        pass
    peak = props.multi_processor_count * 128 * 2 * clock_mhz * 1e6 if clock_mhz else None
    res = {"shape": {"B": B, "Hq": Hq, "Hkv": Hkv, "D": D, "T": T, "key_len": T}, "dtype": "bf16",
           "ms_median": med, "ms_min": best, "fp32_flop": flop, "TFLOPs": flop / med / 1e9,
           "cuda_core_fp32_peak_TFLOPs": peak / 1e12 if peak else None,
           "fraction_of_cuda_core_peak": flop / med / 1e-3 / peak if peak else None,
           "attentions_path_bytes": L * B * Hq * T * T * 2}
    if with_attentions:
        a = torch.softmax(torch.randn(B, Hq, T, T, generator=g, device="cuda"), -1).to(dt)
        ma = manager(L, Hq)
        ma.update_attention_scores([a])
        torch.cuda.synchronize()
        res["attentions_ms_median"] = events(lambda: ma.update_attention_scores([a]), reps)[0]
        del a
    return res


def tpot(tokens, rounds):
    from transformers import DynamicCache, GPTNeoXConfig, GPTNeoXForCausalLM

    from kvcompress.evaluate_attention import evaluate_with_attention_compression

    cfg = GPTNeoXConfig(vocab_size=50304, hidden_size=2560, num_hidden_layers=32, num_attention_heads=32,
                        intermediate_size=10240, max_position_embeddings=2048, rotary_pct=0.25)
    torch.manual_seed(0)
    with torch.device("cuda"):
        model = GPTNeoXForCausalLM(cfg).to(torch.bfloat16).eval()
    ids = torch.randint(0, cfg.vocab_size, (1, tokens), device="cuda")
    # skip_layers=[]: HF sizes the eager mask from layer 0, which would be longer than a compressed layer's keys
    kw = dict(start_size=4, heavy_hitter_size=64, recent_size=444, skip_layers=[], show_progress=False,
              cache="slab", input_ids=ids)

    def run(scores):
        model.set_attn_implementation("eager" if scores == "attentions" else "sdpa")
        m = H2OScoreSlab(start_size=4, heavy_hitter_size=64, recent_size=444, num_layers=32, num_heads=32)
        r = evaluate_with_attention_compression(model, h2o_manager=m, scores=scores, **kw)
        return r["tpot"] * 1e3, r["perplexity"]

    def forwards(impl, out_attn, steps=64):
        model.set_attn_implementation(impl)
        cache = DynamicCache()
        with torch.inference_mode():
            model(ids[:, :512], past_key_values=cache, use_cache=True)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                model(ids[:, 512 + i:513 + i], past_key_values=cache, use_cache=True, output_attentions=out_attn)
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    res = {"eager_output_attentions_scoreslab_ms": [], "capture_queries_sdpa_scoreslab_ms": [], "ppl": {}}
    run("attentions"), run("queries")   # warm-up
    for _ in range(rounds):
        for key, scores in (("eager_output_attentions_scoreslab_ms", "attentions"),
                            ("capture_queries_sdpa_scoreslab_ms", "queries")):
            t, ppl = run(scores)
            res[key].append(t)
            res["ppl"][scores] = ppl
    res["uncompressed_forward_ms_eager_output_attentions_at_512"] = forwards("eager", True)
    res["uncompressed_forward_ms_sdpa_at_512"] = forwards("sdpa", False)
    res["model"] = "Pythia-2.8B-shaped GPT-NeoX, random weights, bf16, batch 1, cache='slab', h2o 4/64/444, no skipped layer"
    res["tokens"] = tokens
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_h2o_query_step.json"))
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--tokens", type=int, default=600)
    ap.add_argument("--skip-tpot", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("h2o_query_step.py measures on a CUDA device; none is visible")
    result = {"gpu": gpu_info(), "torch": torch.__version__, "library": _engine.load_library().kvc_build_info().decode(),
              "peak_reference": "data-sheet 7.7 TB/s HBM3e (HGX B200, one GPU, 1000 W) — not a measured peak"}
    result["update"] = {n: update_alone(n, args.rounds, args.reps) for n in UPDATE_SHAPES}
    result["prefill"] = {str(T): prefill(T, max(3, args.reps // 4), T == 4096) for T in (4096, 16384)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:   # the kernel numbers survive a failure of the end-to-end part
        json.dump(result, f, indent=1)
    if not args.skip_tpot:
        result["tpot"] = tpot(args.tokens, max(2, args.rounds // 2))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"gpu": result["gpu"],
                      "update": {n: {k: round(v[k], 4) for k in ("queries_ms_median", "queries_fraction_of_datasheet",
                                                                  "attentions_ms_median")}
                                 for n, v in result["update"].items()},
                      "prefill": {n: {k: v[k] for k in ("ms_median", "TFLOPs", "fraction_of_cuda_core_peak")}
                                  for n, v in result["prefill"].items()},
                      "tpot": {k: v for k, v in result.get("tpot", {}).items() if k.endswith("ms") or "forward" in k}}))


if __name__ == "__main__":
    main()
