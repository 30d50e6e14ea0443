"""Cumulative H2O (H2OScoreSlab(carry_scores=True)) against the reset semantics, one decode step, on the GPU.

Steady state at the two shapes of scripts/h2o_step.py (bf16), every path timed alternately in one process:
  reset_slab   update, KVSlabCache.compress_ with the same attentions handed over again, reset, append one row per
               layer (the harness's step with the reference's semantics)
  carry_slab   update once, compress_ carrying the accumulators, append (no reset, no second update)
  reset_fn / carry_fn   the same two steps through h2o_attention_compress (gather into fresh tensors)
ms per step from CUDA events and from the host clock around steps that end in a synchronise.

The compaction kernel alone, with and without carry:
  fused (function path): one kvc_compress_layers(_carry) launch on fixed inputs, CUDA events over many launches;
  slab (in place): kvc_slab_compress_kernel's device time in a torch.profiler trace of the two slab steps (a separate
  run: tracing slows the host, not the kernels).
The accumulator bytes a carry moves (read + write of the Hq x C entries of every layer) are computed from the shapes.

    python scripts/h2o_carry_step.py --out profiles/r05_h2o_carry_step.json
"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs3602-llm-inference-acceleration_b200"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

import kvcompress  # noqa: E402
from kvcompress import H2OScoreSlab, KVSlabCache, _engine  # noqa: E402
from kvcompress.methods._common import cached_plans  # noqa: E402
from kvcompress import _planner as P  # noqa: E402
from h2o_step import SHAPES, gpu_info  # noqa: E402


def _median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def time_paths(paths, rounds, steps):
    for fn in paths.values():  # warm-up: modules, plan caches, buffers
        for _ in range(5):
            fn()
    torch.cuda.synchronize()
    host, dev, launches = {k: [] for k in paths}, {k: [] for k in paths}, {}
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
    return {k: {"ms_per_step_events_median": _median(dev[k]), "ms_per_step_events_min": min(dev[k]),
                "ms_per_step_host_median": _median(host[k]), "library_launches_per_step": launches[k]} for k in paths}


def decode(name, rounds, steps, kernel_reps):
    L, B, Hq, Hkv, D, S, start, hh, recent = SHAPES[name]
    dt = torch.bfloat16
    g = torch.Generator(device="cuda").manual_seed(0)
    kv = [(torch.randn(B, Hkv, S, D, generator=g, device="cuda").to(dt),
           torch.randn(B, Hkv, S, D, generator=g, device="cuda").to(dt)) for _ in range(L)]
    attn = [torch.softmax(2 * torch.randn(B, Hq, 1, S, generator=g, device="cuda"), -1).to(dt) for _ in range(L)]
    kw = dict(start_size=start, heavy_hitter_size=hh, recent_size=recent, skip_layers=[])
    mk = dict(start_size=start, heavy_hitter_size=hh, recent_size=recent, num_layers=L, num_heads=Hq)
    m = {k: H2OScoreSlab(**mk, carry_scores=k.startswith("carry")) for k in ("reset_slab", "carry_slab", "reset_fn",
                                                                            "carry_fn")}
    slabs = {k: KVSlabCache.from_legacy_cache(kv, capacity=S + 8) for k in ("reset_slab", "carry_slab")}
    new = [(k[:, :, :1].contiguous(), v[:, :, :1].contiguous()) for k, v in kv]

    def reset_slab():
        m["reset_slab"].update_attention_scores(attn, [])
        slabs["reset_slab"].compress_("h2o_attention", attention_scores=attn, h2o_manager=m["reset_slab"], **kw)
        m["reset_slab"].reset()
        slabs["reset_slab"].append(new)

    def carry_slab():
        m["carry_slab"].update_attention_scores(attn, [])
        slabs["carry_slab"].compress_("h2o_attention", h2o_manager=m["carry_slab"], **kw)
        slabs["carry_slab"].append(new)

    def reset_fn():
        m["reset_fn"].update_attention_scores(attn, [])
        kvcompress.h2o_attention_compress(kv, attention_scores=attn, h2o_manager=m["reset_fn"], **kw)
        m["reset_fn"].reset()

    def carry_fn():
        m["carry_fn"].update_attention_scores(attn, [])
        kvcompress.h2o_attention_compress(kv, h2o_manager=m["carry_fn"], **kw)

    steps_res = time_paths({"reset_slab": reset_slab, "carry_slab": carry_slab, "reset_fn": reset_fn,
                            "carry_fn": carry_fn}, rounds, steps)

    # the fused compaction alone: the same plans and score rows, with and without the carry record
    mgr = H2OScoreSlab(**mk, carry_scores=True)
    mgr.update_attention_scores(attn, [])
    plans = cached_plans(P.plan_h2o, [S] * L, start, hh, recent, skip_layers=[])
    ps, given, scores, carry = mgr.compress_plans(plans, start, hh, recent, B, Hkv, dt, kv[0][0].device)
    C = ps.plans[0].out_len
    variants = {"fused_no_carry": lambda: _engine.run_plans(kv, ps, given_indices=given, given_scores=scores),
                "fused_carry": lambda: _engine.run_plans(kv, ps, given_indices=given, given_scores=scores, carry=carry)}
    for fn in variants.values():
        fn()
    torch.cuda.synchronize()
    fused = {k: [] for k in variants}
    for _ in range(rounds):
        for key, fn in variants.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(kernel_reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            fused[key].append(e0.elapsed_time(e1) * 1e3 / kernel_reps)
    fused = {k: {"us_per_launch_events_median": _median(v), "us_per_launch_events_min": min(v)} for k, v in fused.items()}

    # the in-place compaction alone: kernel device time from a trace of the two slab steps
    slab_kernel = {}
    for key, fn in (("slab_no_carry", reset_slab), ("slab_carry", carry_slab)):
        with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
            for _ in range(steps):
                fn()
            torch.cuda.synchronize()
        t = [e.device_time_total for e in prof.events()
             if e.device_type == torch.autograd.DeviceType.CUDA and "kvc_slab_compress_kernel" in e.name]
        slab_kernel[key] = {"us_per_launch_median": _median(t), "us_per_launch_min": min(t), "launches": len(t)}
    acc_bytes = 2 * L * B * Hq * C * 2   # read + write of every carried bf16 accumulator entry
    return {"shape": dict(zip(("L", "B", "Hq", "Hkv", "D", "S", "start", "heavy_hitters", "recent"), SHAPES[name])),
            "dtype": "bf16", "C": C, "rounds": rounds, "steps_per_round": steps, "decode_step": steps_res,
            "fused_kernel": fused, "slab_kernel_profiler": slab_kernel, "carried_accumulator_bytes": acc_bytes}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_h2o_carry_step.json"))
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--kernel-reps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("h2o_carry_step.py measures on a CUDA device; none is visible")
    result = {"gpu": gpu_info(), "torch": torch.__version__, "library": _engine.load_library().kvc_build_info().decode(),
              "decode": {name: decode(name, args.rounds, args.steps, args.kernel_reps) for name in SHAPES}}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    summary = {n: {"step_ms": {k: round(v["ms_per_step_events_median"], 3) for k, v in d["decode_step"].items()},
                   "fused_us": {k: round(v["us_per_launch_events_median"], 1) for k, v in d["fused_kernel"].items()},
                   "slab_us": {k: round(v["us_per_launch_median"], 1) for k, v in d["slab_kernel_profiler"].items()}}
               for n, d in result["decode"].items()}
    print(json.dumps({"gpu": result["gpu"], "summary": summary}))


if __name__ == "__main__":
    main()
