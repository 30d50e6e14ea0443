"""Beam search's per-step cache reorder on the GPU: KVSlabCache.reorder_ (one kvc_batch_reorder launch for K, V, the
key norms of every layer and the followers' state) against the reorder transformers runs on a DynamicCache today
(Cache.reorder_cache: index_select of K and V per layer, 2 x L launches and allocations).

Shapes: Pythia-2.8B (32 layers, 32 heads, head_dim 80, bf16, 4 beams) and Llama-3-8B GQA (32 layers, 8 KV heads of 32
query heads, head_dim 128, bf16, 8 beams), every layer at 512, 1024 or 4096 rows, with an H2OScoreSlab (accumulators
of every layer at the same length) and a full 32-row SnapKVQueryWindow as followers.  Indices: a typical beam step
(entry b takes b - b % 2: half the entries move, each source twice) and a full permutation (a rotation by one).

Per case: kernel time from CUDA events around `--calls` back-to-back calls (median of `--rounds`), the bytes the
reorder needs (each distinct source read once, each moving destination written once), GB/s and the share of the copy
peak of MEASURED_PEAKS.json when present (else of the data-sheet 7.7 TB/s, named as such); the DynamicCache reorder
timed the same way.  Working sets of the 512-row Pythia cases fit the 126 MB L2 in part; the rest do not.

    python scripts/slab_reorder_step.py --out profiles/r08_slab_reorder.json
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "cs3602-llm-inference-acceleration_b200"))
sys.path.insert(0, os.path.join(ROOT, "scripts"))
import torch  # noqa: E402

from h2o_step import DATASHEET_TBPS, gpu_info, measured_hbm_peak  # noqa: E402
from kvcompress import H2OScoreSlab, KVSlabCache, SnapKVQueryWindow, _engine  # noqa: E402

MODELS = {
    # name: layers, KV heads, query heads, head_dim, beams
    "pythia2.8b": (32, 32, 32, 80, 4),
    "llama3_8b_gqa": (32, 8, 32, 128, 8),
}
LENGTHS = (512, 1024, 4096)
W = 32


def sm_clock():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=clocks.sm", "--format=csv,noheader"], capture_output=True,
                              text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:
        return f"unavailable ({e})"


def time_calls(fn, calls, rounds):
    fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(rounds):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(calls):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 1e-3 / calls)
    return sorted(out)[len(out) // 2]


def case(model, S, kind, calls, rounds, peak):
    L, Hkv, Hq, D, B = MODELS[model]
    dt, e = torch.bfloat16, 2
    slab = KVSlabCache(L, B, Hkv, D, S, dt)
    for t in (slab.k, slab.v, slab.n):
        t.normal_()
    slab.lengths = [S] * L
    h2o = H2OScoreSlab(num_layers=L, num_heads=Hq, capacity=S)
    h2o._ensure(B, Hq, dt, slab.device, S)
    h2o._acc.normal_()
    h2o._lens = {l: S for l in range(L)}
    win = SnapKVQueryWindow(L, B, Hq, D, W, dt)
    win._buf.normal_()
    win.filled = [W] * L
    idx = [b - b % 2 for b in range(B)] if kind == "beam" else [(b + 1) % B for b in range(B)]
    moving = [b for b in range(B) if idx[b] != b]
    sources = len({idx[b] for b in moving})
    entry = L * (2 * Hkv * S * D * e + Hkv * S * e + Hq * S * e + Hq * W * D * e)  # one batch entry's valid bytes
    nbytes = (sources + len(moving)) * entry
    index = torch.tensor(idx, device="cuda")
    n0 = _engine.launch_count()
    slab.reorder_(index, h2o, win)
    launches = _engine.launch_count() - n0
    t = time_calls(lambda: slab.reorder_(index, h2o, win), calls, rounds)
    # transformers' reorder of a DynamicCache holding the same K and V (no norms, no followers)
    keys = [slab[l][0].contiguous() for l in range(L)]
    values = [slab[l][1].contiguous() for l in range(L)]
    del slab, h2o, win

    def hf():
        for l in range(L):
            keys[l] = keys[l].index_select(0, index)
            values[l] = values[l].index_select(0, index)

    t_hf = time_calls(hf, calls, rounds)
    hf_bytes = 2 * B * L * 2 * Hkv * S * D * e
    del keys, values
    torch.cuda.empty_cache()
    return {"model": model, "rows": S, "beams": B, "index": kind, "index_values": idx, "launches": launches,
            "bytes_moved": nbytes, "kernel_s": t, "GBps": nbytes / t / 1e9, "share_of_copy_peak": nbytes / t / peak,
            "hf_dynamic_cache": {"launches": 2 * L, "s": t_hf, "bytes_read_and_written_kv_only": hf_bytes,
                                 "GBps": hf_bytes / t_hf / 1e9}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_slab_reorder.json"))
    ap.add_argument("--calls", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("slab_reorder_step.py measures on a CUDA device; none is visible")
    peak, label, raw = measured_hbm_peak(os.path.join(ROOT, "MEASURED_PEAKS.json"))
    if peak is None:
        peak, label = DATASHEET_TBPS * 1e12, "data-sheet 7.7 TB/s (HGX B200, one GPU, 1000 W) - not a measured peak"
    result = {"gpu": dict(gpu_info(), sm_clock_at_start=sm_clock()), "torch": torch.__version__,
              "library": _engine.load_library().kvc_build_info().decode(), "peak_reference": label,
              "measured_peaks_file": raw, "calls_per_round": args.calls, "rounds": args.rounds, "cases": []}
    for model in MODELS:
        for S in LENGTHS:
            for kind in ("beam", "permutation"):
                r = case(model, S, kind, args.calls, args.rounds, peak)
                result["cases"].append(r)
                print(f"{model} S={S} {kind}: {r['kernel_s'] * 1e6:.1f} us, {r['bytes_moved'] / 1e6:.0f} MB, "
                      f"{r['GBps']:.0f} GB/s ({r['share_of_copy_peak']:.2f} of peak), launches {r['launches']}; "
                      f"DynamicCache {r['hf_dynamic_cache']['s'] * 1e6:.1f} us", flush=True)
    result["gpu"]["sm_clock_at_end"] = sm_clock()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
