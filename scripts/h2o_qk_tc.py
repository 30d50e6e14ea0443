"""The H2O query update on the tensor cores (H2OScoreSlab(tensor_cores=True), kvc_h2o_accumulate_qk_tc) against the
CUDA-core form (kvc_h2o_accumulate_qk) on one GPU.

  prompt   one layer, Hq 32, Hkv 8, D 128, bf16, B 1, T = key_len in {1024, 4096, 16384, 32768} (the CUDA-core form is
           skipped at 32768): CUDA-event medians over alternating rounds of the two forms in one process; per pass
           (statistics, column sums, score row) the kernel times of one profiled call, run separately.  Rates: the
           MMA work 2 * 2 * D per visible (query, key) pair (both passes) against the data-sheet 2250 TFLOP/s dense
           bf16, and the exponentials (one per visible pair and pass) against the ex2 rate scripts/lab/ex2_mix_bw.cu
           measures on the same card for the vote's pass-2 loop (ex2 / clk / SM x SMs x max SM clock).
  decode   the two decode shapes of scripts/h2o_query_step.py that fit one update: Pythia-2.8B B 1 at 513 keys and
           Llama-3-8B GQA B 8 at 1025 keys, 32 layers, one query per step, both forms.
  e2e      a 32-layer Pythia-2.8B-shaped random-weight bf16 GPT-NeoX on a 4096-token prompt under capture_queries: the
           H2O prefill update of all layers from the captured q and K, each form.

    python scripts/h2o_qk_tc.py --out profiles/r06_h2o_qk_tc.json
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs3602-llm-inference-acceleration_b200"))
import torch  # noqa: E402

import kvcompress  # noqa: E402
from kvcompress import H2OScoreSlab, _engine  # noqa: E402

DATASHEET_BF16_TFLOPS = 2250.0
DECODE_SHAPES = {
    # name: L, B, Hq, Hkv, D, key_len
    "pythia2.8b_b1_s513": (32, 1, 32, 32, 80, 513),
    "llama3_8b_gqa_b8_s1025": (32, 8, 32, 8, 128, 1025),
}


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "sms": torch.cuda.get_device_properties(0).multi_processor_count}


def ex2_rate(gpu):
    """ex2 per second: the ex2 / clk / SM that scripts/lab/ex2_mix_bw.cu (built in a temporary directory) measures for the
    vote's pass-2 loop, x SMs x the max SM clock."""
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "ex2_mix_bw")
        subprocess.run(["nvcc", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                        os.path.join(ROOT, "scripts", "lab", "ex2_mix_bw.cu")], check=True, capture_output=True)
        text = subprocess.run([exe], check=True, capture_output=True, text=True, timeout=300).stdout
    # the vote kernel's pass-2 loop: ffma -> ex2 -> fadd fed from TMEM and shared memory, as this kernel's pass 2 (the
    # first line's loop has operands that never change and reads 8x the other three)
    per_clk = float(re.search(r"both.*?([0-9.]+) ex2 / clk / SM", text).group(1))
    mhz = float(gpu["max_sm_clock"].split()[0])
    return {"ex2_per_clk_per_sm": per_clk, "ex2_per_s": per_clk * gpu["sms"] * mhz * 1e6, "lab_output": text.strip()}


def events(fn, reps):
    out = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    out.sort()
    return out[len(out) // 2]


def manager(L, Hq, tc):
    return H2OScoreSlab(start_size=4, heavy_hitter_size=64, recent_size=444, num_layers=L, num_heads=Hq,
                        tensor_cores=tc)


def per_pass(fn):
    """Kernel time per pass of one call, from the profiler (a run of its own)."""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        if ev.device_type == torch.autograd.DeviceType.CUDA:
            n = ev.name
            key = ("statistics" if ("Lb0E" in n or "false>" in n) else "column_sums") if "h2o_tc_kernel" in n else \
                "stats" if "qk_stats" in n else "accumulate" if "qk_accumulate" in n else \
                "score_row" if "h2o_accumulate_kernel" in n else n[:60]
            out[key] = round(out.get(key, 0.0) + ev.device_time_total / 1e3, 4)  # ms
    return out


def compare(fns, rounds, reps):
    for fn in fns.values():
        fn()
    torch.cuda.synchronize()
    med = {k: [] for k in fns}
    for _ in range(rounds):   # alternate the forms
        for k, fn in fns.items():
            med[k].append(events(fn, reps))
    return {k: sorted(v)[len(v) // 2] for k, v in med.items()}


def prompt(T, rounds, reps, ex2, with_cuda_core):
    B, Hq, Hkv, D = 1, 32, 8, 128
    g = torch.Generator(device="cuda").manual_seed(1)
    keys = [torch.randn(B, Hkv, T, D, generator=g, device="cuda").bfloat16()]
    qs = [(2 * torch.randn(B, Hq, T, D, generator=g, device="cuda")).bfloat16()]
    m_tc, m_cc = manager(1, Hq, True), manager(1, Hq, False)
    fns = {"tensor_cores": lambda: m_tc.update_from_queries(qs, keys)}
    if with_cuda_core:
        fns["cuda_cores"] = lambda: m_cc.update_from_queries(qs, keys)
    ms = compare(fns, rounds, reps)
    pairs = B * Hq * T * (T + 1) // 2            # visible (query, key) pairs of the causal rule
    flop_pass = 2 * D * pairs
    passes = per_pass(fns["tensor_cores"])
    res = {"shape": {"B": B, "Hq": Hq, "Hkv": Hkv, "D": D, "T": T, "key_len": T}, "dtype": "bf16",
           "ms_median": ms, "visible_pairs": pairs, "tc_kernel_ms": passes,
           "tc_TFLOPs_both_passes": 2 * flop_pass / ms["tensor_cores"] / 1e9,
           "tc_exp_per_s": 2 * pairs / ms["tensor_cores"] * 1e3}
    for p in ("statistics", "column_sums"):
        if passes.get(p):
            res[f"tc_{p}_TFLOPs"] = flop_pass / passes[p] / 1e9
            res[f"tc_{p}_fraction_of_datasheet_mma"] = flop_pass / passes[p] / 1e9 / DATASHEET_BF16_TFLOPS
            res[f"tc_{p}_fraction_of_ex2_rate"] = pairs / passes[p] * 1e3 / ex2["ex2_per_s"]
    if with_cuda_core:
        res["speedup"] = ms["cuda_cores"] / ms["tensor_cores"]
        res["cc_kernel_ms"] = per_pass(fns["cuda_cores"])
    return res


def decode(name, rounds, reps):
    L, B, Hq, Hkv, D, S = DECODE_SHAPES[name]
    g = torch.Generator(device="cuda").manual_seed(0)
    keys = [torch.randn(B, Hkv, S, D, generator=g, device="cuda").bfloat16() for _ in range(L)]
    qs = [(2 * torch.randn(B, Hq, 1, D, generator=g, device="cuda")).bfloat16() for _ in range(L)]
    m_tc, m_cc = manager(L, Hq, True), manager(L, Hq, False)
    fns = {"tensor_cores": lambda: m_tc.update_from_queries(qs, keys),
           "cuda_cores": lambda: m_cc.update_from_queries(qs, keys)}
    launches = {}
    for k, fn in fns.items():
        n0 = _engine.launch_count()
        fn()
        launches[k] = _engine.launch_count() - n0
    ms = compare(fns, rounds, reps)
    return {"shape": dict(zip(("L", "B", "Hq", "Hkv", "D", "key_len"), DECODE_SHAPES[name])), "dtype": "bf16",
            "launches_per_update": launches, "ms_median": ms, "tc_kernel_ms": per_pass(fns["tensor_cores"]),
            "cc_kernel_ms": per_pass(fns["cuda_cores"])}


def e2e(tokens, reps):
    from transformers import GPTNeoXConfig, GPTNeoXForCausalLM

    cfg = GPTNeoXConfig(vocab_size=50304, hidden_size=2560, num_hidden_layers=32, num_attention_heads=32,
                        intermediate_size=10240, max_position_embeddings=tokens, rotary_pct=0.25)
    torch.manual_seed(0)
    with torch.device("cuda"):
        model = GPTNeoXForCausalLM(cfg).to(torch.bfloat16).eval()
    model.set_attn_implementation("sdpa")
    ids = torch.randint(0, cfg.vocab_size, (1, tokens), device="cuda")
    with torch.inference_mode():
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        model(ids, use_cache=True)
        e0.record()
        model(ids, use_cache=True)
        e1.record()
        torch.cuda.synchronize()
        forward_ms = e0.elapsed_time(e1)
        with kvcompress.capture_queries(model) as cap:
            model(ids, use_cache=True)
    args = (cap.queries, cap.keys, cap.masks, cap.scaling)
    m_tc, m_cc = manager(32, 32, True), manager(32, 32, False)
    ms = compare({"tensor_cores": lambda: (m_tc.reset(), m_tc.update_from_queries(*args)),
                  "cuda_cores": lambda: (m_cc.reset(), m_cc.update_from_queries(*args))}, 1, reps)
    return {"model": "Pythia-2.8B-shaped GPT-NeoX (32 layers, Hq 32, D 80), random weights, bf16, batch 1, SDPA",
            "tokens": tokens, "masks_recorded": sum(m is not None for m in cap.masks),
            "h2o_prefill_update_ms_median": ms, "speedup": ms["cuda_cores"] / ms["tensor_cores"],
            "model_forward_ms": forward_ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_h2o_qk_tc.json"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-e2e", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("h2o_qk_tc.py measures on a CUDA device; none is visible")
    gpu = gpu_info()
    result = {"gpu": gpu, "torch": torch.__version__, "library": _engine.load_library().kvc_build_info().decode(),
              "peak_reference": f"data-sheet {DATASHEET_BF16_TFLOPS} TFLOP/s dense bf16 (HGX B200, one GPU, 1000 W) — not "
                                "a measured peak; ex2 rate measured on this card by scripts/lab/ex2_mix_bw.cu"}
    result["ex2"] = ex2_rate(gpu)
    result["prompt"] = {str(T): prompt(T, args.rounds, args.reps if T <= 4096 else 3, result["ex2"], T <= 16384)
                        for T in (1024, 4096, 16384, 32768)}
    result["decode"] = {n: decode(n, args.rounds, 4 * args.reps) for n in DECODE_SHAPES}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:   # the kernel numbers survive a failure of the end-to-end part
        json.dump(result, f, indent=1)
    if not args.skip_e2e:
        result["e2e"] = e2e(4096, 3)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps({"gpu": gpu, "prompt": {T: v["ms_median"] for T, v in result["prompt"].items()},
                      "decode": {n: v["ms_median"] for n, v in result["decode"].items()},
                      "e2e": result.get("e2e", {}).get("h2o_prefill_update_ms_median")}))


if __name__ == "__main__":
    main()
