"""H2O with attention scores, one decode step and one prefill-sized accumulate, on the GPU.

Decode steady state (the attention-score harness's step: update, compress with a second update of the same
attentions, reset), three paths timed alternately in one process:
  (a) H2OAttentionManager + h2o_attention_compress  (torch bookkeeping; it refuses batch > 1, so at B > 1 the step
      runs once per batch entry — what a user has to do with it)
  (b) H2OScoreSlab + h2o_attention_compress
  (c) H2OScoreSlab + KVSlabCache.compress_            (the step also appends one row per layer to the slab)
ms per step from the host clock around steps that end in a synchronise, and from CUDA events; a torch.profiler kernel
list of one step of (c).

Prefill-sized accumulate: one kvc_h2o_accumulate over 32 layers of [1, 32, 2048, 2048] bf16 attention probabilities
(8.6 GB, far beyond L2), achieved bytes/s against MEASURED_PEAKS.json when present, else the data-sheet 7.7 TB/s.

    python scripts/h2o_step.py --out profiles/r03_h2o_step.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs3602-llm-inference-acceleration_b200"))
import torch  # noqa: E402

import kvcompress  # noqa: E402
from kvcompress import H2OAttentionManager, H2OScoreSlab, KVSlabCache, _engine  # noqa: E402

SHAPES = {
    # name: L, B, Hq, Hkv, D, S (= budget + 1), start, heavy hitters, recent
    "pythia2.8b_b1": (32, 1, 32, 32, 80, 513, 4, 64, 444),
    "llama3_8b_gqa_b8": (32, 8, 32, 8, 128, 1025, 4, 64, 956),
}
DATASHEET_TBPS = 7.7


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:  # the measurement still names the device through torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": f"unavailable ({e})"}


def decode_paths(name, rounds, steps):
    L, B, Hq, Hkv, D, S, start, hh, recent = SHAPES[name]
    dt = torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(0)
    kv = [(torch.randn(B, Hkv, S, D, generator=g, device="cuda").to(dt),
           torch.randn(B, Hkv, S, D, generator=g, device="cuda").to(dt)) for _ in range(L)]
    attn = [torch.softmax(2 * torch.randn(B, Hq, 1, S, generator=g, device="cuda"), -1).to(dt) for _ in range(L)]
    kw = dict(start_size=start, heavy_hitter_size=hh, recent_size=recent, skip_layers=[])
    mk = dict(start_size=start, heavy_hitter_size=hh, recent_size=recent, num_layers=L, num_heads=Hq)
    m_torch, m_fn, m_slab = H2OAttentionManager(**mk), H2OScoreSlab(**mk), H2OScoreSlab(**mk)
    slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
    new = [(k[:, :, :1].contiguous(), v[:, :, :1].contiguous()) for k, v in kv]
    per_entry = [([(k[b:b + 1], v[b:b + 1]) for k, v in kv], [a[b:b + 1] for a in attn]) for b in range(B)]

    def step_a():
        for kv_b, attn_b in per_entry:
            m_torch.update_attention_scores(attn_b, [])
            kvcompress.h2o_attention_compress(kv_b, attention_scores=attn_b, h2o_manager=m_torch, **kw)
            m_torch.reset()

    def step_b():
        m_fn.update_attention_scores(attn, [])
        kvcompress.h2o_attention_compress(kv, attention_scores=attn, h2o_manager=m_fn, **kw)
        m_fn.reset()

    def step_c():
        m_slab.update_attention_scores(attn, [])
        slab.compress_("h2o_attention", attention_scores=attn, h2o_manager=m_slab, **kw)
        m_slab.reset()
        slab.append(new)

    paths = {"a_torch_manager_function": step_a, "b_scoreslab_function": step_b, "c_scoreslab_slab_compress": step_c}
    # the same kept rows on every path (batch entry 0, every layer)
    outs = {}
    m_torch.update_attention_scores(per_entry[0][1], [])
    outs["a"] = kvcompress.h2o_attention_compress(per_entry[0][0], attention_scores=per_entry[0][1],
                                                  h2o_manager=m_torch, **kw)
    m_torch.reset()
    m_fn.update_attention_scores(attn, [])
    outs["b"] = kvcompress.h2o_attention_compress(kv, attention_scores=attn, h2o_manager=m_fn, **kw)
    m_fn.reset()
    same = all(torch.equal(outs["a"][l][0], outs["b"][l][0][:1]) and torch.equal(outs["a"][l][1], outs["b"][l][1][:1])
               for l in range(L))
    for fn in paths.values():  # warm-up: modules, plan caches, buffers
        for _ in range(5):
            fn()
    torch.cuda.synchronize()
    host = {k: [] for k in paths}
    dev = {k: [] for k in paths}
    launches = {}
    for _ in range(rounds):
        for key, fn in paths.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            n0 = _engine.launch_count()
            t0 = time.perf_counter()
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            host[key].append((time.perf_counter() - t0) * 1e3 / steps)
            dev[key].append(e0.elapsed_time(e1) / steps)
            launches[key] = (_engine.launch_count() - n0) / steps
    res = {}
    for key in paths:
        h, d = sorted(host[key]), sorted(dev[key])
        res[key] = {"ms_per_step_host_median": h[len(h) // 2], "ms_per_step_host_min": h[0],
                    "ms_per_step_events_median": d[len(d) // 2], "library_launches_per_step": launches[key]}
    # one step of (c) under the profiler
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        step_c()
        torch.cuda.synchronize()
    kernels = [{"name": e.name[:120], "us": round(e.device_time_total, 2)} for e in prof.events()
               if e.device_type == torch.autograd.DeviceType.CUDA]
    return {"shape": dict(zip(("L", "B", "Hq", "Hkv", "D", "S", "start", "heavy_hitters", "recent"), SHAPES[name])),
            "dtype": "bf16", "rounds": rounds, "steps_per_round": steps, "paths": res,
            "kept_rows_equal_a_b_entry0": same, "profiler_kernels_one_step_c": kernels}


def measured_hbm_peak(path):
    """(bytes/s, label, file contents) of the first HBM / bandwidth entry of MEASURED_PEAKS.json, or (None, None, ...)."""
    if not os.path.exists(path):
        return None, None, None
    raw = json.load(open(path))

    def walk(d, prefix=""):
        for k, v in (d.items() if isinstance(d, dict) else []):
            if isinstance(v, dict):
                yield from walk(v, prefix + k + ".")
            elif isinstance(v, (int, float)):
                yield prefix + k, float(v)

    for key, v in walk(raw):
        low = key.lower()
        if ("hbm" in low or "bandwidth" in low or "copy" in low) and v > 0:
            scale = 1.0 if v > 1e11 else (1e9 if v > 100 else 1e12)  # bytes/s, GB/s or TB/s
            return v * scale, f"MEASURED_PEAKS.json:{key}", raw
    return None, None, raw


def prefill_accumulate(reps):
    L, B, H, Q = 32, 1, 32, 2048
    dt = torch.bfloat16
    attn = torch.empty((L, B, H, Q, Q), dtype=dt, device="cuda").uniform_(0, 1e-3)
    layers = list(attn.unbind(0))
    m = H2OScoreSlab(start_size=4, heavy_hitter_size=64, recent_size=444, num_layers=L, num_heads=H)
    m.update_attention_scores(layers)   # warm-up, allocation; later calls decay + add (prev_len = key_len)
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        m.update_attention_scores(layers)
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1) * 1e-3)
    # bytes the algorithm needs: attention read once, accumulators read and written, the score rows written
    e = 2
    attn_bytes = L * B * H * Q * Q * e
    acc_bytes = 2 * L * B * H * Q * e
    score_bytes = L * B * (Q - 444 - 4) * e
    total = attn_bytes + acc_bytes + score_bytes
    best, med = min(times), sorted(times)[len(times) // 2]
    peak_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_label, raw = measured_hbm_peak(peak_path)
    if peak is None:
        peak = DATASHEET_TBPS * 1e12
        peak_label = "data-sheet 7.7 TB/s (HGX B200, one GPU, 1000 W) — not a measured peak"
    return {"measured_peaks_file": raw, "shape": {"L": L, "B": B, "Hq": H, "n_query": Q, "key_len": Q}, "dtype": "bf16", "reps": reps,
            "bytes": total, "attention_bytes": attn_bytes, "kernel_s_median": med, "kernel_s_min": best,
            "achieved_TBps_median": total / med / 1e12, "achieved_TBps_best": total / best / 1e12,
            "fraction_of_peak_median": total / med / peak, "peak_reference": peak_label}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_h2o_step.json"))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--prefill-reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("h2o_step.py measures on a CUDA device; none is visible")
    result = {"gpu": gpu_info(), "torch": torch.__version__, "library": _engine.load_library().kvc_build_info().decode(),
              "decode": {name: decode_paths(name, args.rounds, args.steps) for name in SHAPES},
              "prefill_accumulate": prefill_accumulate(args.prefill_reps)}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    summary = {n: {k: round(v["ms_per_step_host_median"], 3) for k, v in d["paths"].items()}
               for n, d in result["decode"].items()}
    print(json.dumps({"gpu": result["gpu"], "decode_ms_host_median": summary,
                      "prefill_TBps_median": round(result["prefill_accumulate"]["achieved_TBps_median"], 3),
                      "prefill_fraction_of_peak": round(result["prefill_accumulate"]["fraction_of_peak_median"], 3)}))


if __name__ == "__main__":
    main()
