#!/usr/bin/env python
"""bench.py — the compress-step benchmark (BASELINE.json metric) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config c2] [--impl ours|reference] [--dump-outputs DIR]

One *step* = one pass of the compress hot path over one batch of synthetic KV cache: every call the
config names (for the default c2: ``streaming_llm_compress(4, 508)`` then
``fix_size_l2_compress(512, 0.2, keep_low)``) on a Pythia-2.8B-shaped bf16 cache, batch 32, 4K
context, resident in HBM.  ``value`` = algorithmic bytes of a step (e*B*H*D*(R + 4C) per compressed
layer, SURVEY.md §8d) / device time, summed over ranks; weak scaling (each rank owns 32 streams).

The printed JSON line follows the driver contract and adds

* ``roofline``  the dominant kernel against the measured HBM copy peak;
* ``e2e``       the same step on a HOST-resident cache (pinned ``KVSlabCache``: K, V and the key norms recorded at
                append time) through the public compress functions, PCIe traffic inside the timed region;
* ``cpu_baseline`` the C port of the reference's algorithm (oracle/kvc_oracle.c, OpenMP) on a bounded sample, with
                the UNMODIFIED reference's own torch code (baseline/_ref, ``scripts/install_ref.sh``) timed beside it
                on the host CPU and on the B200 (``cpu_baseline_reference`` / ``eager_gpu``);
* ``configs``   every other BASELINE.json configuration (c1, c2 steady state, c3, c4, c4 vote, c5, batch 1), a few
                timed steps each, per call: microseconds, GB/s, fraction of the measured peak;
* ``strong``    BASELINE configs[2] and [4] as GLOBAL jobs (c3: B = 256 at 8K; c5: B = 64 at 32K, once batch-sharded
                and once layer-sharded) split over the N ranks, sequential slabs where a rank's share exceeds HBM,
                with a checksum of the kept indices that is independent of N.

``--impl reference`` times the CPU port alone on all host threads.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "cs3602-llm-inference-acceleration_b200"))

PYTHIA = dict(model_shape="pythia-2.8b", L=32, H=32, D=80)
LLAMA = dict(model_shape="llama-3-8b-gqa", L=32, H=8, D=128)
CONFIGS = {
    # BASELINE.json configs[1] — the configuration the metric is quoted on (fits one GPU: 42.9 GB)
    "c2": dict(PYTHIA, B=32, S=4096, dtype="bf16", calls=[
        ("streaming_llm", dict(start_size=4, recent_size=508)),
        ("fix_size_l2", dict(fix_kv_size=512, keep_ratio=0.2, strategy="keep_low")),
    ]),
    # the same two calls at decode steady state (S = cap + 1)
    "c2_steady": dict(PYTHIA, B=32, S=513, dtype="bf16", calls=[
        ("streaming_llm", dict(start_size=4, recent_size=508)),
        ("fix_size_l2", dict(fix_kv_size=512, keep_ratio=0.2, strategy="keep_low")),
    ]),
    # configs[2]: B=256 total = 8 ranks x 32 streams (86 GB per rank)
    "c3": dict(PYTHIA, B=32, S=8192, dtype="bf16", calls=[
        ("h2o_l2", dict(start_size=4, heavy_hitter_size=64, recent_size=444)),
    ]),
    # configs[3]
    "c4": dict(LLAMA, B=16, S=32768, dtype="bf16", calls=[
        ("snapkv_lite", dict(observation_window=32, keep_size=512)),
    ]),
    # configs[3] with the opt-in tcgen05 q.K^T vote (4 query heads per KV head, W=32 -> 128 query rows)
    "c4_vote": dict(LLAMA, B=16, S=32768, dtype="bf16", calls=[
        ("snapkv_lite", dict(observation_window=32, keep_size=512, _vote_group=4)),
    ]),
    # the same with the window queries' log-sum-exp supplied by the caller (an attention forward returns it):
    # the kernel skips its first pass and reads K once
    "c4_vote_lse": dict(LLAMA, B=16, S=32768, dtype="bf16", calls=[
        ("snapkv_lite", dict(observation_window=32, keep_size=512, _vote_group=4, _vote_lse=True)),
    ]),
    # the vote on an MHA model: Pythia shape, one query head per KV head (32 of the 128 query rows in use)
    "c2_vote": dict(PYTHIA, B=32, S=4096, dtype="bf16", calls=[
        ("snapkv_lite", dict(observation_window=32, keep_size=512, _vote_group=1)),
    ]),
    # configs[4]: B=64 total = 8 ranks x 8 streams (34 GB per rank)
    "c5": dict(LLAMA, B=8, S=32768, dtype="bf16", calls=[
        ("pyramid_kv", dict(base_size=512)),
        ("adaptive_l2", dict(target_size=512)),
    ]),
    # configs[0] on the GPU for reference: fp32, batch 1
    "c1": dict(PYTHIA, B=1, S=2048, dtype="f32", calls=[
        ("l2_compress", dict(keep_ratio=0.8, prune_after=1000, skip_layers=[0, 1])),
    ]),
}
FALLBACK_HBM_GBS = 6650.0  # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--config", default="c2", choices=sorted(CONFIGS))
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="override the per-rank batch")
    ap.add_argument("--seq-len", type=int, default=0, help="override the context length (diagnostics)")
    ap.add_argument("--mode", default="functions", choices=["functions", "slab"],
                    help="functions: the drop-in compress functions (default, the BASELINE metric); slab: the same calls "
                         "in place on a KVSlabCache (append + compress_), SURVEY 8f rank 1")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config table (c1 ... c5, batch 1)")
    ap.add_argument("--no-strong", action="store_true", help="skip the strong-scaling section (global c3 / c5 jobs)")
    ap.add_argument("--no-eager", action="store_true", help="skip the reference-torch comparator legs")
    ap.add_argument("--table-steps", type=int, default=5, help="timed steps per entry of the configs table")
    ap.add_argument("--sustain-s", type=float, default=1.5,
                    help="configs table, c4 / c4_vote / c4_vote_lse: seconds of back-to-back calls for the sustained row")
    ap.add_argument("--e2e-slab", type=int, default=8, help="streams per host<->device slab in the e2e leg")
    ap.add_argument("--cpu-sample-batch", type=int, default=0,
                    help="streams in the CPU sample (0: enough (b,h) rows to occupy every host thread, at most 8)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write what the last timed step returned (rank 0) to DIR/*.npy as float32, so that two builds "
                         "can be compared output for output; see dump_outputs()")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.mode != "functions"):
        ap.error("--dump-outputs writes the outputs of the compress functions (--impl ours --mode functions)")
    return args


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def profiled_traffic(config: str):
    """dram read+write bytes per launch of the dominant kernel from the committed ncu capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(config)
    except Exception:
        return None


# --------------------------------------------------------------------------- plans / bytes
def plans_for(method, seq_lens, kw):
    from kvcompress import _planner as P

    kw = dict(kw)
    if method == "streaming_llm":
        return P.plan_streaming(seq_lens, kw.get("start_size", 4), kw.get("recent_size", 508), kw.get("skip_layers", []))
    if method == "fix_size_l2":
        return P.plan_fix_size(seq_lens, kw.get("fix_kv_size", 1024), kw.get("keep_ratio", 0.0),
                               kw.get("strategy", "keep_low"), kw.get("skip_layers", [0, 1]))
    if method == "h2o_l2":
        return P.plan_h2o(seq_lens, kw.get("start_size", 4), kw.get("heavy_hitter_size", 64), kw.get("recent_size", 444),
                          kw.get("skip_layers", []))
    if method == "snapkv_lite":
        return P.plan_snapkv(seq_lens, kw.get("observation_window", 32), kw.get("keep_size", 512),
                             kw.get("pooling_kernel", 5), kw.get("skip_layers", []))
    if method == "pyramid_kv":
        return P.plan_pyramid(seq_lens, kw.get("base_size", 512), kw.get("layer_decay", 0.9), kw.get("min_size", 64),
                              kw.get("profile", "exponential"), kw.get("skip_layers", []))
    if method == "adaptive_l2":
        return P.plan_adaptive(seq_lens, kw.get("target_size", 512), kw.get("soft_limit", 256),
                               kw.get("hard_limit", 1024), kw.get("keep_ratio_min", 0.3), kw.get("keep_ratio_max", 0.9),
                               kw.get("skip_layers", []))
    if method == "l2_compress":
        return P.plan_l2(seq_lens, kw.get("keep_ratio", 1.0), kw.get("prune_after", 1000), kw.get("skip_layers", [0, 1]))
    raise KeyError(method)


def call_bytes(cfg, batch):
    from kvcompress import _planner as P

    e = 4 if cfg["dtype"] == "f32" else 2
    out = []
    for method, kw in cfg["calls"]:
        plans = plans_for(method, [cfg["S"]] * cfg["L"], kw)
        nbytes = P.algorithmic_bytes(plans, batch, cfg["H"], cfg["D"], e)
        if "_vote_group" in kw and not kw.get("_vote_lse"):
            # vote mode reads the region's K rows twice (SURVEY 8d: e*B*H*D*(2R + 4C)); once when the caller holds the LSE
            nbytes += sum(p.region for p in plans if p.kind == P.GATHER) * batch * cfg["H"] * cfg["D"] * e
        out.append(nbytes)
    return out


# --------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """SM clock + throttle reasons DURING the timed region, sampled in-process through NVML every few
    milliseconds (the timed region is tens of milliseconds: an `nvidia-smi -lms` child would not even
    have started).  Same fields as the profiling recipe's nvidia-smi line."""

    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"),
               ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"),
               ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"),
               ("hw_power_brake", "nvmlClocksEventReasonHwPowerBrakeSlowdown"))

    def __init__(self, cuda_index: int, period_s: float = 0.002):
        self.cuda_index = cuda_index
        self.period_s = period_s
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.power_w = []
        self._stop = None
        self._thread = None
        self._err = None

    def _handle(self, nv):
        import torch

        try:  # CUDA_VISIBLE_DEVICES renumbers CUDA devices; NVML does not — go through the UUID
            uuid = str(torch.cuda.get_device_properties(self.cuda_index).uuid)
            return nv.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            return nv.nvmlDeviceGetHandleByIndex(self.cuda_index)

    def start(self):
        import threading

        try:
            import pynvml as nv

            nv.nvmlInit()
            h = self._handle(nv)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
        except Exception as exc:  # no NVML: report empty clocks rather than fail the bench
            self._err = repr(exc)
            return
        self._stop = threading.Event()

        def loop():
            while not self._stop.is_set():
                try:
                    self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                    for name, attr in self.REASONS:
                        if mask & getattr(nv, attr):
                            self.reasons.add(name)
                    self.power_w.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                except Exception as exc:
                    self._err = repr(exc)
                    return
                self._stop.wait(self.period_s)

        self._thread = threading.Thread(target=loop, daemon=True)
        self._thread.start()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        if self._thread is not None:
            self._stop.set()
            self._thread.join(timeout=5)
        if self.samples:
            out["sm_mhz"] = statistics.median(self.samples)
            out["sm_mhz_min"] = min(self.samples)
            out["samples"] = len(self.samples)
            out["power_w_max"] = round(max(self.power_w), 1) if self.power_w else None
        out["reasons"] = sorted(self.reasons)
        out["how"] = "NVML in-process, every 2 ms, during the timed region only"
        if self._err:
            out["error"] = self._err
        return out


# --------------------------------------------------------------------------- synthetic cache
def make_cache(cfg, batch, device, seed):
    """BASELINE.md §3 spread-norm synthetic cache, generated on the device, layer by layer."""
    import torch

    dt = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}[cfg["dtype"]]
    H, S, D = cfg["H"], cfg["S"], cfg["D"]
    kv = []
    for layer in range(cfg["L"]):
        g = torch.Generator(device=device).manual_seed(seed + layer)
        k = torch.randn(batch, H, S, D, generator=g, device=device)
        k *= torch.exp(0.35 * torch.randn(batch, H, S, 1, generator=g, device=device))
        k[:, :, :4] *= 0.1
        v = torch.randn(batch, H, S, D, generator=g, device=device)
        kv.append((k.to(dt), v.to(dt)))
        del k, v
    return kv


# --------------------------------------------------------------------------- CPU port (oracle) leg
def cpu_sample_batch(cfg, requested, cap):
    from oracle import kvc_oracle_c as OC

    if requested > 0:
        return min(requested, cap)
    return max(1, min(cap, 8, max(2, -(-OC.max_threads() // cfg["H"]))))


def cpu_port_run(cfg, sample_batch, steps, warmup, host_layers=None, threads=0, min_seconds=0.0):
    """Time oracle/kvc_oracle.c (the reference's algorithm, OpenMP over (b,h)) on a bounded sample: `steps` timed
    passes, extended until `min_seconds` of CPU work have been timed (at most 400 passes)."""
    import numpy as np
    import torch

    from oracle import kvc_oracle as O
    from oracle import kvc_oracle_c as OC

    threads = threads or OC.max_threads()
    dtype = cfg["dtype"]
    if host_layers is None:
        tdt = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}[dtype]
        g = torch.Generator().manual_seed(1234)
        host_layers = []
        for _ in range(cfg["L"]):
            k = torch.randn(sample_batch, cfg["H"], cfg["S"], cfg["D"], generator=g)
            k *= torch.exp(0.35 * torch.randn(sample_batch, cfg["H"], cfg["S"], 1, generator=g))
            k[:, :, :4] *= 0.1
            v = torch.randn(sample_batch, cfg["H"], cfg["S"], cfg["D"], generator=g)
            host_layers.append((k.to(tdt), v.to(tdt)))

    def as_np(t):
        return t.view(torch.int16).numpy().view(np.uint16) if dtype == "bf16" else t.numpy()

    layers = [(as_np(k), as_np(v)) for k, v in host_layers]
    e = 4 if dtype == "f32" else 2
    step_bytes = 0
    for method, kw in cfg["calls"]:
        step_bytes += O.algorithmic_bytes(O.METHODS[method](layers, dtype, select=None,
                                                            **{k: v for k, v in kw.items() if not k.startswith("_")}), e)
    times = []
    it = 0
    while True:
        t = 0.0
        for method, kw in cfg["calls"]:
            _, _, dt_s = OC.run_method(method, layers, dtype, nthreads=threads,
                                       **{k: v for k, v in kw.items() if not k.startswith("_")})
            t += dt_s
        if it >= warmup:
            times.append(t)
        it += 1
        if len(times) >= steps and (sum(times) >= min_seconds or len(times) >= 400):
            break
    mean_s = sum(times) / len(times)
    return dict(gbs=step_bytes / mean_s / 1e9, seconds_per_step=mean_s, threads=threads, step_bytes=step_bytes,
                sample=f"{cfg['L']} layers x (B={sample_batch}, H={cfg['H']}, S={cfg['S']}, D={cfg['D']}) {dtype}, "
                       f"{len(times)} timed passes of the same calls ({sum(times):.1f} s of CPU work)")


# --------------------------------------------------------------------------- the UNMODIFIED reference (baseline/_ref)
def load_reference():
    """The reference's own package, copied unmodified by scripts/install_ref.sh to baseline/_ref/kvcompress_ref.
    Returns its COMPRESS_METHODS dict, or (None, why)."""
    ref_root = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_root, "kvcompress_ref")):
        return None, "baseline/_ref/kvcompress_ref is absent (run scripts/install_ref.sh where /root/reference exists)"
    if ref_root not in sys.path:
        sys.path.insert(0, ref_root)
    try:
        from kvcompress_ref.methods import COMPRESS_METHODS as ref_methods
    except Exception as exc:  # the reference needs transformers
        return None, f"import failed: {exc!r}"
    return ref_methods, None


def reference_torch_run(cfg, layers, steps, warmup, min_seconds=0.0, max_steps=50):
    """Time the reference's own functions (stock code path: torch.norm -> argsort -> sort -> gather -> cat per layer)
    on `layers` (CPU tensors: host cores; CUDA tensors: the B200).  Returns dict or {'unavailable': why}."""
    import torch

    ref_methods, why = load_reference()
    if ref_methods is None:
        return {"unavailable": why}
    on_gpu = layers[0][0].is_cuda
    calls = [(ref_methods[m], {k: v for k, v in kw.items() if not k.startswith("_")}) for m, kw in cfg["calls"]]
    B = layers[0][0].size(0)
    step_bytes = sum(call_bytes(cfg, B))
    times = []
    it = 0
    with torch.inference_mode():
        while True:
            if on_gpu:
                torch.cuda.synchronize()
            t0 = time.perf_counter()
            for fn, kw in calls:
                out = fn(layers, **kw)
            if on_gpu:
                torch.cuda.synchronize()
            dt_s = time.perf_counter() - t0
            del out
            if it >= warmup:
                times.append(dt_s)
            it += 1
            if len(times) >= steps and (sum(times) >= min_seconds or len(times) >= max_steps):
                break
    mean_s = sum(times) / len(times)
    return {"value": round(step_bytes / mean_s / 1e9, 3), "unit": "GB/s", "kind": "reference",
            "ms_per_sample_step": round(mean_s * 1e3, 3),
            "cores": torch.get_num_threads() if not on_gpu else None,
            "sample": f"{cfg['L']} layers x (B={B}, H={cfg['H']}, S={cfg['S']}, D={cfg['D']}) {cfg['dtype']}, "
                      f"{len(times)} timed passes ({sum(times):.1f} s) of the reference's own functions on "
                      f"{'cuda' if on_gpu else 'the host CPU'} (baseline/_ref/kvcompress_ref, unmodified)"}


# --------------------------------------------------------------------------- reference arm
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    cfg = dict(CONFIGS[args.config])
    steps = max(1, args.steps)
    warmup = max(0, args.warmup)
    sb = cpu_sample_batch(cfg, args.cpu_sample_batch or 8, cfg["B"])  # 8 streams: ~0.5 s per pass on 16 cores
    res = cpu_port_run(cfg, sb, steps, warmup)  # exactly `steps` timed passes of the bounded sample
    # the reference's own torch code on the same host cores, a smaller sample (it is several times slower)
    ref_line = None
    if not args.no_eager:
        tdt = {"bf16": torch.bfloat16, "f16": torch.float16, "f32": torch.float32}[cfg["dtype"]]
        g = torch.Generator().manual_seed(1234)
        pair = [(torch.randn(2, cfg["H"], cfg["S"], cfg["D"], generator=g).to(tdt),
                 torch.randn(2, cfg["H"], cfg["S"], cfg["D"], generator=g).to(tdt)) for _ in range(2)]
        small = [pair[l % 2] for l in range(cfg["L"])]  # the functions never mutate their input: layers may share storage
        torch.set_num_threads(os.cpu_count() or 1)
        ref_line = reference_torch_run(cfg, small, steps=2, warmup=1, min_seconds=5.0)
    line = {
        "impl": "reference", "metric": "kv_compress_step_throughput", "value": round(res["gbs"], 3), "unit": "GB/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
        "ms_per_step": round(res["seconds_per_step"] * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
        # the SAME config as the repo arm's line (contract: "on your arm's config"); what was actually timed per step is
        # the bounded sample described in cpu_baseline.sample
        "config": workload_config(cfg, args.config, cfg["B"], max(1, args.gpus)),
        "cpu_baseline": {"value": round(res["gbs"], 3), "unit": "GB/s", "cores": res["threads"], "kind": "port",
                         "sample": res["sample"]},
        "cpu_baseline_reference": ref_line,
        "e2e": {"value": round(res["gbs"], 3), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "the reference is pure Python on torch (no native sources to compile): this arm's value is the C port "
                "of its algorithm (oracle/kvc_oracle.c: norm -> full sort -> take k -> sort -> gather, OpenMP over "
                "(batch, head)) on all host threads — the FASTER of the two CPU baselines; the reference's own torch "
                "functions on the same cores are in cpu_baseline_reference.  The sample is a batch slice (B="
                f"{sb} of {cfg['B']} streams: throughput in GB/s does not depend on it) because the full cache does not "
                "fit host memory next to its outputs.",
    }
    print(json.dumps(line), flush=True)


def workload_config(cfg, name, batch, n_gpus):
    calls = "; ".join(f"{m}({', '.join(f'{k}={v}' for k, v in kw.items())})" for m, kw in cfg["calls"])
    return {
        "workload": f"{name}: {calls} on a synthetic {cfg['model_shape']}-shaped {cfg['dtype']} KV cache, "
                    f"{cfg['L']} layers x (B={batch}, H={cfg['H']}, S={cfg['S']}, D={cfg['D']}) per GPU",
        "global_batch": batch * n_gpus, "seq_len": cfg["S"], "layers": cfg["L"], "kv_heads": cfg["H"],
        "head_dim": cfg["D"], "parallelism": f"batch-sharded x{n_gpus}, no collective on the hot path",
        "l2_policy": "inputs (>= 5 GB per step) are far larger than the 126 MB L2; no explicit flush",
    }


def bind_to_gpu_cpus(cuda_index: int):
    """Multi-rank runs: bind this rank to the CPU cores nearest its GPU (NVML's ideal affinity) before any pinned
    host buffer is allocated, so the e2e leg's host cache is first-touched on the GPU's NUMA node and the ranks
    do not all pull from one socket.  Returns a description of what happened (never None: a failure says why)."""
    before = len(os.sched_getaffinity(0))
    try:
        import pynvml as nv
        import torch

        nv.nvmlInit()
        uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
        h = nv.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
        nv.nvmlDeviceSetCpuAffinity(h)
        after = sorted(os.sched_getaffinity(0))
        return {"bound": True, "cores_before": before, "cores_after": len(after), "first_core": after[0],
                "last_core": after[-1], "how": "nvmlDeviceSetCpuAffinity (ideal affinity of this rank's GPU)"}
    except Exception as exc:
        return {"bound": False, "cores_before": before, "why": repr(exc)}


# --------------------------------------------------------------------------- timing a config's calls
def vote_inputs(cfg, B, kv, device):
    """Synthetic observation-window queries [B, H*G, W, D] per layer for the vote configs (and, for the single-pass
    variant, their log-sum-exp, computed the way an attention forward would)."""
    import math

    import torch

    extra = {}
    flops = 0
    g = torch.Generator(device=device).manual_seed(5678)   # the same queries on every run
    for m, kw in cfg["calls"]:
        if "_vote_group" not in kw:
            continue
        G, Wn = kw["_vote_group"], kw["observation_window"]
        qs = [(1.5 * torch.randn(B, cfg["H"] * G, Wn, cfg["D"], generator=g, device=device)).to(kv[0][0].dtype)
              for _ in range(cfg["L"])]
        extra["obs_queries"] = qs
        passes = 1 if kw.get("_vote_lse") else 2
        flops += passes * 2 * 128 * cfg["S"] * cfg["D"] * B * cfg["H"] * cfg["L"]  # 128 = padded query rows of the MMA
        if kw.get("_vote_lse"):
            lses = []
            S, P = cfg["S"], cfg["S"] - Wn
            for (k, _), q in zip(kv, qs):
                out = torch.empty(B, cfg["H"] * G, Wn, device=device, dtype=torch.float32)
                for b in range(B):  # one stream at a time: [H*G, W, S] fp32 scores
                    kk = k[b].float().repeat_interleave(G, dim=0)
                    sc = torch.matmul(q[b].float(), kk.transpose(-1, -2)) / math.sqrt(cfg["D"])
                    pos_q = P + torch.arange(Wn, device=device).view(1, Wn, 1)
                    sc.masked_fill_(torch.arange(S, device=device).view(1, 1, S) > pos_q, float("-inf"))
                    out[b] = torch.logsumexp(sc, dim=-1)
                lses.append(out)
            extra["obs_lse"] = lses
    return extra, flops


def time_calls(cfg, B, kv, steps, warmup, device, barrier=None, sampler=None, back_to_back=0, sustain_s=0.0,
               outputs=None):
    """`steps` timed passes of the config's calls on `kv` (CUDA events on torch's current stream = the launch stream).
    Returns (total_ms, per_call list of dicts, launches, vote_flops).  `outputs` (a list) receives what each call of
    the last timed pass returned."""
    import torch

    import kvcompress
    from kvcompress import _engine

    per_call_bytes = call_bytes(cfg, B)
    extra, vote_flops = vote_inputs(cfg, B, kv, device)
    fns = []
    for m, kw in cfg["calls"]:
        run_kw = {k: v for k, v in kw.items() if not k.startswith("_")}
        if "_vote_group" in kw:
            run_kw.update(extra)
        fns.append((kvcompress.get_compress_fn(m), run_kw))
    torch.cuda.synchronize()

    def one_step(events=None, keep=None):
        for i, (fn, kw) in enumerate(fns):
            if events is not None:
                events[i][0].record()
            out = fn(kv, **kw)
            if events is not None:
                events[i][1].record()
            if keep is not None:
                keep.append(out)
            del out

    for _ in range(warmup):
        one_step()
    if barrier:
        barrier()
    else:
        torch.cuda.synchronize()
    ev = [[(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in fns] for _ in range(steps)]
    t_begin, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler is not None:
        sampler.start()
        if barrier:
            barrier()
    launches0 = _engine.launch_count()
    t_wall = time.perf_counter()
    t_begin.record()
    for s in range(steps):
        one_step(ev[s], outputs if s == steps - 1 else None)
    t_end.record()
    if barrier:
        barrier()
    else:
        torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t_wall) * 1e3
    launches = _engine.launch_count() - launches0
    total_ms = t_begin.elapsed_time(t_end)
    peak, _ = measured_peak()
    per_call = []
    for i, (m, _) in enumerate(cfg["calls"]):
        ms = [ev[s][i][0].elapsed_time(ev[s][i][1]) for s in range(steps)]
        mean = statistics.mean(ms)
        per_call.append({"call": m, "us_mean": round(mean * 1e3, 1), "us_min": round(min(ms) * 1e3, 1),
                         "algorithmic_bytes": per_call_bytes[i],
                         "gbs": round(per_call_bytes[i] / (mean * 1e-3) / 1e9, 1),
                         "frac_of_peak": round(per_call_bytes[i] / (mean * 1e-3) / 1e9 / peak, 4)})
    if back_to_back:
        # latency-bound shapes (batch 1): the calls queued back to back with no event in between — what a decode loop
        # sees when the GPU already has work queued — timed once around the whole train
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for _ in range(back_to_back):
            one_step()
        b.record()
        host_us = (time.perf_counter() - t0) * 1e6 / (back_to_back * len(fns))
        torch.cuda.synchronize()
        wall_us = (time.perf_counter() - t0) * 1e6 / (back_to_back * len(fns))
        dev_us = a.elapsed_time(b) * 1e3 / (back_to_back * len(fns))
        per_call.append({"call": "back_to_back", "calls": back_to_back * len(fns), "host_us_per_call": round(host_us, 1),
                         "wall_us_per_call": round(wall_us, 1), "device_us_per_call": round(dev_us, 1),
                         "gbs": round(sum(per_call_bytes) / len(fns) / dev_us / 1e3, 1),
                         "frac_of_peak": round(sum(per_call_bytes) / len(fns) / dev_us / 1e3 / peak, 4),
                         "us_mean": round(dev_us, 1), "us_min": round(dev_us, 1), "algorithmic_bytes": sum(per_call_bytes) // len(fns)})
    if sustain_s > 0:
        # the timed steps above are a burst of a few calls; a kernel that needs SM cycles (the vote) slows down once
        # the board settles at its power limit: the same calls back to back for `sustain_s` seconds, NVML beside them
        torch.cuda.synchronize()
        smp = ClockSampler(device.index or 0, period_s=0.005)
        smp.start()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0, n = time.perf_counter(), 0
        a.record()
        while time.perf_counter() - t0 < sustain_s:
            for _ in range(4):
                one_step()
            n += 4
            torch.cuda.synchronize()
        b.record()
        torch.cuda.synchronize()
        clk = smp.stop()
        dev_us = a.elapsed_time(b) * 1e3 / (n * len(fns))
        per_call.append({"call": "sustained", "calls": n * len(fns), "seconds": round(time.perf_counter() - t0, 2),
                         "us_mean": round(dev_us, 1), "us_min": round(dev_us, 1),
                         "algorithmic_bytes": sum(per_call_bytes) // len(fns),
                         "gbs": round(sum(per_call_bytes) / len(fns) / dev_us / 1e3, 1),
                         "frac_of_peak": round(sum(per_call_bytes) / len(fns) / dev_us / 1e3 / peak, 4),
                         "sm_mhz": clk.get("sm_mhz"), "sm_mhz_min": clk.get("sm_mhz_min"),
                         "power_w_max": clk.get("power_w_max"), "clock_reasons": clk.get("reasons")})
    return total_ms, per_call, launches, vote_flops, wall_ms


def time_in_place(cfg, B, kv, steps, device):
    """The config's calls IN PLACE on a KVSlabCache holding the same rows (stored key norms instead of the K scan, kept
    rows slide down inside the slab): per call the mean / min device time of `compress_` over `steps` runs.  A
    prefill-sized compress is re-armed by rewinding the slab's lengths (timing does not depend on the values)."""
    import torch

    from kvcompress import KVSlabCache

    S, rows = cfg["S"], []
    per_call_bytes = call_bytes(cfg, B)
    for i, (method, kw) in enumerate(cfg["calls"]):
        run_kw = {k: v for k, v in kw.items() if not k.startswith("_")}
        slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
        ms = []
        for step in range(steps + 2):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            slab.compress_(method, **run_kw)
            b.record()
            torch.cuda.synchronize()
            slab.lengths = [S] * cfg["L"]
            if step >= 2:
                ms.append(a.elapsed_time(b))
        rows.append({"call": method, "us_mean": round(statistics.mean(ms) * 1e3, 1), "us_min": round(min(ms) * 1e3, 1),
                     "speedup_over_function": None,
                     "effective_gbs": round(per_call_bytes[i] / (statistics.mean(ms) * 1e-3) / 1e9, 1)})
        del slab
        torch.cuda.empty_cache()
    return rows


def configs_table(args, device):
    """Every other BASELINE configuration on this GPU, a few timed steps each (driver-visible copies of the numbers
    DESIGN.md quotes).  Caches are generated and freed one config at a time."""
    import torch

    table = {}
    order = [("c2_steady", None), ("c2_steady_b1", ("c2_steady", 1)), ("c1", None), ("c3", None), ("c5", None),
             ("c4", None), ("c4_vote", None), ("c4_vote_lse", None), ("c2_vote", None)]
    sustained = ("c4", "c4_vote", "c4_vote_lse")  # measured LAST: seconds at the power limit would colour later bursts
    kv, kv_key = None, None
    steps = max(2, args.table_steps)
    for name, alias in order:
        base, B = (alias if alias else (name, None))
        cfg = dict(CONFIGS[base])
        B = B or cfg["B"]
        key = (cfg["model_shape"], B, cfg["S"], cfg["dtype"])
        t0 = time.perf_counter()
        try:
            if key != kv_key:  # c4 / c4_vote / c4_vote_lse share one cache
                kv = None
                torch.cuda.empty_cache()
                kv = make_cache(cfg, B, device, seed=4321)
                kv_key = key
            sampler = ClockSampler(device.index or 0)
            total_ms, per_call, launches, vote_flops, wall_ms = time_calls(
                cfg, B, kv, steps, 2, device, None, sampler, back_to_back=50 if B == 1 else 0)
            clk = sampler.stop()
            entry = {"workload": workload_config(cfg, base, B, 1)["workload"], "steps": steps,
                     "sm_mhz": clk.get("sm_mhz"), "clock_reasons": clk.get("reasons"),
                     "ms_per_step": round(total_ms / steps, 4), "wall_ms_per_step": round(wall_ms / steps, 4),
                     "per_call": per_call, "gpu_launches": launches,
                     "min_frac_of_peak": min(c["frac_of_peak"] for c in per_call
                                             if c["call"] not in ("back_to_back", "sustained"))}
            if vote_flops:
                entry["tensor_tflops"] = round(vote_flops / (total_ms / steps * 1e-3) / 1e12, 1)
            prof = profiled_traffic(name) if B == cfg["B"] else None
            if prof and prof.get("per_call"):  # DRAM bytes per launch from the committed ncu captures
                for c in per_call:
                    if c["call"] in prof["per_call"]:
                        c["traffic"] = prof["per_call"][c["call"]]
                entry["traffic_source"] = prof["source"]
            if B == 1:
                entry["note"] = ("batch 1: the per-call rows time ONE call between two events on an idle GPU (launch latency "
                                 "included); the back_to_back row is the same calls queued without events")
            if name in ("c2_steady", "c2_steady_b1", "c4", "c5"):  # the cache and a slab copy of it fit next to each other
                try:
                    entry["in_place"] = {"what": "the same calls as KVSlabCache.compress_ on a slab holding the same rows "
                                                 "(scores from the stored key norms, kept rows slide down in place); "
                                                 "effective_gbs = the function's algorithmic bytes / this time",
                                         "per_call": time_in_place(cfg, B, kv, steps, device)}
                    fn_us = {c["call"]: c["us_mean"] for c in per_call}
                    for r in entry["in_place"]["per_call"]:
                        r["speedup_over_function"] = round(fn_us[r["call"]] / r["us_mean"], 2) if r["call"] in fn_us else None
                except Exception as exc:
                    entry["in_place"] = {"error": repr(exc)[:300]}
        except Exception as exc:  # one config failing must not take the headline line with it
            entry = {"error": repr(exc)[:300]}
            kv, kv_key = None, None
            torch.cuda.empty_cache()
        entry["seconds_incl_setup"] = round(time.perf_counter() - t0, 1)
        table[name] = entry
    if args.sustain_s > 0:
        for name in sustained:  # the three share one cache
            cfg = dict(CONFIGS[name])
            if "error" in table.get(name, {"error": 1}):
                continue
            try:
                key = (cfg["model_shape"], cfg["B"], cfg["S"], cfg["dtype"])
                if key != kv_key:
                    kv = None
                    torch.cuda.empty_cache()
                    kv = make_cache(cfg, cfg["B"], device, seed=4321)
                    kv_key = key
                _, rows, _, _, _ = time_calls(cfg, cfg["B"], kv, 1, 1, device, None, None, sustain_s=args.sustain_s)
                table[name]["per_call"] += [r for r in rows if r["call"] == "sustained"]
            except Exception as exc:
                table[name]["sustained_error"] = repr(exc)[:300]
    kv = None
    torch.cuda.empty_cache()
    return table


# --------------------------------------------------------------------------- strong scaling (global c3 / c5 jobs)
def fill_block(k, v, seed, dt):
    """Spread-norm synthetic rows (BASELINE.md §3) written into existing tensors; the same seed gives the same bytes
    on every rank, whichever rank owns the block."""
    import torch

    g = torch.Generator(device=k.device).manual_seed(seed)
    k.normal_(generator=g)            # in place: no slab-sized temporaries, the allocator's blocks stay as they are
    scale = torch.exp(0.35 * torch.randn(k.shape[:-1] + (1,), generator=g, device=k.device)).to(dt)
    scale[:, :, :4] *= 0.1
    k.mul_(scale)
    v.normal_(generator=g)


def idx_checksum(indices):
    """Order-sensitive checksum of kept rows: sum over layers of sum(idx * (position + 1)), python int."""
    import torch

    total = 0
    for li in sorted(indices):
        idx = indices[li].long()
        w = torch.arange(1, idx.size(-1) + 1, device=idx.device)
        total += int((idx * w).sum().item()) * (li + 1)
    return total


def strong_section(args, device, world, rank, barrier):
    """BASELINE configs[2] (c3: h2o_l2, B = 256 at 8K, 687 GB) and configs[4] (c5: pyramid_kv + adaptive_l2, B = 64 at
    32K, 275 GB) as GLOBAL jobs split over the ranks: c3 and c5 batch-sharded (kvcompress.sharding.shard_range over
    blocks of streams), c5 also layer-sharded (shard_layers, per-layer budget table replicated).  A rank walks its
    share as sequential slabs of one resident buffer (a slab = what fits HBM: 86 GB for c3, 34 GB for c5), each
    slab regenerated from seeds keyed by (layer, stream block), so the kept-index checksum summed over ranks is the
    same at every N.  Timed: CUDA events around each slab's compress calls; global step = max over ranks."""
    import torch
    import torch.distributed as dist

    from kvcompress import _engine, _planner, sharding

    dt = torch.bfloat16
    out = {}
    jobs = [
        ("c3_batch", "c3", 256, 32, "batch"),    # 8 blocks of 32 streams, all layers
        ("c5_batch", "c5", 64, 8, "batch"),      # 8 blocks of 8 streams, all layers
        ("c5_layer", "c5", 64, 8, "layer"),      # 8 groups of 4 layers, all 64 streams (8 blocks of 8 per layer)
    ]
    for name, base, global_B, block_B, how in jobs:
        cfg = dict(CONFIGS[base])
        L, H, S, D = cfg["L"], cfg["H"], cfg["S"], cfg["D"]
        n_blocks = global_B // block_B
        t_setup = time.perf_counter()
        try:
            plans_all = [plans_for(m, [S] * L, kw) for m, kw in cfg["calls"]]  # global per-layer budgets, every rank
            units = sharding.job_units(how, L, n_blocks, world, rank, layer_group=4)
            slab_layers = max((len(u[0]) for u in units), default=0)
            slab_B = block_B * max((len(u[1]) for u in units), default=0)
            torch.cuda.empty_cache()
            buf = [(torch.empty(slab_B, H, S, D, device=device, dtype=dt), torch.empty(slab_B, H, S, D, device=device, dtype=dt))
                   for _ in range(slab_layers)]
            my_ms = first_ms = 0.0
            checksum = 0
            slabs = 0
            if units:  # untimed first call: the output blocks come out of torch's caching allocator afterwards
                for (k, v) in buf[:len(units[0][0])]:
                    k.zero_(), v.zero_()
                for plans in plans_all:
                    warm = _engine.PlanSet([plans[l] for l in units[0][0]])
                    _engine.run_plans(buf[:len(units[0][0])], warm)
                    _engine.run_plans(buf[:len(units[0][0])], warm, return_indices=True)
                torch.cuda.synchronize()
            for layer_ids, block_ids in units:
                kv = buf[:len(layer_ids)]
                for (k, v), l in zip(kv, layer_ids):
                    for j, bb in enumerate(block_ids):   # the same bytes for (layer l, block bb) whoever owns it
                        fill_block(k[j * block_B:(j + 1) * block_B], v[j * block_B:(j + 1) * block_B],
                                   7_000_000 + 1000 * l + bb, dt)
                torch.cuda.synchronize()
                a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                sub = [_engine.PlanSet([plans[l] for l in layer_ids]) for plans in plans_all]
                c2 = torch.cuda.Event(enable_timing=True)
                a.record()
                for ps in sub:      # timed: exactly what the public functions launch (no index output)
                    out_kv = _engine.run_plans(kv, ps)
                    del out_kv
                b2.record()
                for ps in sub:      # the same slab once more, back to back: separates the kernel from whatever the
                    out_kv = _engine.run_plans(kv, ps)   # in-place regeneration left behind (clocks, dirty L2)
                    del out_kv
                c2.record()
                torch.cuda.synchronize()
                first_ms += a.elapsed_time(b2)
                my_ms += b2.elapsed_time(c2)
                slabs += 1
                results = [_engine.run_plans(kv, ps, return_indices=True) for ps in sub]   # untimed: the kept rows
                for ci, (_, idx) in enumerate(results):   # one term per (call, layer, block): independent of the cut
                    for j in range(len(block_ids)):
                        checksum += (ci + 1) * idx_checksum({layer_ids[i]: t[j * block_B:(j + 1) * block_B]
                                                             for i, t in idx.items()})
                del results
            del buf
            torch.cuda.empty_cache()
            stats = torch.tensor([my_ms, first_ms], device=device, dtype=torch.float64)
            csum = torch.tensor([checksum % (1 << 62)], device=device, dtype=torch.int64)
            per_rank = [my_ms]
            if world > 1:
                gathered = [torch.zeros_like(stats) for _ in range(world)]
                dist.all_gather(gathered, stats)
                per_rank = [float(g[0].item()) for g in gathered]
                first_ms = max(float(g[1].item()) for g in gathered)
                parts = [torch.zeros_like(csum) for _ in range(world)]
                dist.all_gather(parts, csum)
                total_sum = sum(int(p.item()) for p in parts) % (1 << 62)
            else:
                total_sum = int(csum.item())
            step_bytes = sum(_planner.algorithmic_bytes(p, global_B, H, D, 2) for p in plans_all)
            global_ms = max(per_rank)
            out[name] = {
                "workload": f"{base} global job: {'; '.join(m for m, _ in cfg['calls'])} on {L} layers x (B={global_B}, H={H}, "
                            f"S={S}, D={D}) bf16 = {2 * L * global_B * H * S * D * 2 / 1e9:.0f} GB of cache, {how}-sharded over "
                            f"{world} rank(s)",
                "ms_per_global_step": round(global_ms, 3), "per_rank_ms": [round(x, 3) for x in per_rank],
                "ms_first_pass_after_regeneration": round(first_ms, 3),
                "slabs_per_rank": slabs, "algorithmic_bytes": step_bytes,
                "gbs": round(step_bytes / (global_ms * 1e-3) / 1e9, 1),
                "kept_index_checksum": total_sum,
                "seconds_incl_setup": round(time.perf_counter() - t_setup, 1),
            }
        except Exception as exc:
            out[name] = {"error": repr(exc)[:300]}
            torch.cuda.empty_cache()
        barrier()
    out["how"] = ("scaling=strong: total work fixed as N grows; per slab the cache is regenerated in place from seeds keyed "
                  "by (layer, stream block) and only the compress calls are timed (CUDA events), twice back to back: "
                  "ms_per_global_step sums the second pass of every slab, ms_first_pass_after_regeneration the first (it "
                  "starts on a GPU that has just run the random-number kernels); kept_index_checksum is "
                  "summed over ranks with NCCL all_gather and must be identical at every N (and between c5_batch and c5_layer)")
    return out


# --------------------------------------------------------------------------- output dump
DUMP_BYTES = 60_000_000  # row data of all files together; the .npy headers and lengths add well under 1 MB


def dump_outputs(out_dir, cfg, outputs):
    """Write what the config's calls returned, one list of (K, V) per call, so that two builds can be compared output
    for output.  Per call `i` and method `m`:

    * `{i}_{m}_out_len.npy`  float64 [L]: rows each layer came back with;
    * `{i}_{m}_k.npy`, `{i}_{m}_v.npy`  float32 [rows, D]: for every layer in turn, a sample of its output rows (the
      (batch, head, position) rows drawn without replacement by numpy's PCG64 seeded with (i, layer), ascending; all
      rows when a layer has fewer), so that the files together stay under 64 MB.  The sample depends only on the
      output shapes: equal lengths mean the same rows are compared."""
    import numpy as np
    import torch

    os.makedirs(out_dir, exist_ok=True)
    n_tensors = sum(2 * len(out) for out in outputs)
    cap = max(1, DUMP_BYTES // (4 * cfg["D"] * n_tensors))   # sampled rows per output tensor
    for i, ((method, _), out) in enumerate(zip(cfg["calls"], outputs)):
        lens, ks, vs = [], [], []
        for li, (k, v) in enumerate(out):
            B, H, S, _ = k.shape
            lens.append(S)
            pick = np.sort(np.random.default_rng([i, li]).choice(B * H * S, size=min(B * H * S, cap), replace=False))
            b, h, s = (torch.from_numpy(x).to(k.device) for x in np.unravel_index(pick, (B, H, S)))
            ks.append(k[b, h, s].float().cpu().numpy())
            vs.append(v[b, h, s].float().cpu().numpy())
        prefix = os.path.join(out_dir, f"{i}_{method}")
        np.save(prefix + "_out_len.npy", np.asarray(lens, dtype=np.float64))
        np.save(prefix + "_k.npy", np.concatenate(ks))
        np.save(prefix + "_v.npy", np.concatenate(vs))


# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import torch
    import torch.distributed as dist

    from kvcompress import _engine

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the compress path has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    binding = bind_to_gpu_cpus(local) if world > 1 else {"bound": False, "why": "single rank: not needed"}
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    _engine.load_library()

    cfg = dict(CONFIGS[args.config])
    if args.seq_len:
        cfg["S"] = args.seq_len
    B = args.batch or cfg["B"]
    step_bytes = sum(call_bytes(cfg, B))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    kv = make_cache(cfg, B, device, seed=1234 + 1000 * rank)
    W = max(args.warmup, 3)
    K = args.steps
    sampler = ClockSampler(local)
    outputs = [] if args.dump_outputs else None
    total_ms, per_call_list, launches, vote_flops, _ = time_calls(cfg, B, kv, K, W, device, barrier, sampler,
                                                                  outputs=outputs)
    clocks = sampler.stop()
    if outputs is not None:
        if rank == 0:
            dump_outputs(args.dump_outputs, cfg, outputs)
        del outputs
    if world > 1:
        t = torch.tensor([total_ms], device=device, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / K
    value = step_bytes * world / (ms_per_step * 1e-3) / 1e9

    # dominant kernel: the call with the most device time
    dom = max(range(len(per_call_list)), key=lambda i: per_call_list[i]["us_mean"])
    peak, peak_src = measured_peak()
    d = per_call_list[dom]
    prof = profiled_traffic(args.config) if (B == CONFIGS[args.config]["B"] and not args.seq_len) else None
    roofline = {
        "bound": "hbm", "kernel": f"kvc_fused_tma_kernel ({d['call']})", "achieved": d["gbs"],
        "peak": peak, "unit": "GB/s", "frac": d["frac_of_peak"], "frac_of_nominal_8000": round(d["gbs"] / 8000.0, 4),
        "peak_source": peak_src, "algorithmic_bytes_per_launch": d["algorithmic_bytes"],
        "launch_us_mean": d["us_mean"], "launch_us_min": d["us_min"],
        "traffic": prof["bytes_per_launch"] if prof else None, "traffic_source": prof["source"] if prof else None,
    }
    per_call = {c["call"]: {k: v for k, v in c.items() if k != "call"} for c in per_call_list}

    # ------------------------------------------------------------------ e2e: host-resident cache
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(cfg, B, kv, step_bytes, args, device, world, barrier)
    # ------------------------------------------------------------------ the reference's own torch code on this GPU
    eager = None
    if not args.no_eager and world == 1:
        try:
            eager = reference_torch_run(cfg, kv, steps=3, warmup=1)
            if "value" in eager:
                eager["speedup_of_value"] = round(value / eager["value"], 1)
        except Exception as exc:
            eager = {"unavailable": repr(exc)[:200]}
        torch.cuda.empty_cache()
    # ------------------------------------------------------------------ CPU baselines (rank 0, N=1)
    cpu, cpu_ref = None, None
    if not args.no_cpu_baseline and world == 1 and rank == 0:
        sb = cpu_sample_batch(cfg, args.cpu_sample_batch, B)
        host_layers = [(k[:sb].cpu(), v[:sb].cpu()) for k, v in kv]
        kv = None
        torch.cuda.empty_cache()
        res = cpu_port_run(cfg, sb, steps=2, warmup=1, host_layers=host_layers, min_seconds=12.0)
        cpu = {"value": round(res["gbs"], 3), "unit": "GB/s", "cores": res["threads"], "kind": "port",
               "sample": res["sample"], "seconds_per_sample_step": round(res["seconds_per_step"], 4)}
        if not args.no_eager:
            torch.set_num_threads(os.cpu_count() or 1)
            cpu_ref = reference_torch_run(cfg, host_layers, steps=2, warmup=1, min_seconds=6.0)
        del host_layers
    elif world > 1:
        cpu = None  # measured on rank 0 at N=1 only (contract); see the N=1 line
    kv = None
    torch.cuda.empty_cache()

    # ------------------------------------------------------------------ every other config; global jobs
    table = None
    if not args.no_configs and world == 1 and args.config == "c2" and not args.batch and not args.seq_len:
        table = configs_table(args, device)
    strong = None
    if not args.no_strong and args.config == "c2" and not args.batch and not args.seq_len:
        strong = strong_section(args, device, world, rank, barrier)

    if rank == 0:
        line = {
            "metric": "kv_compress_step_throughput", "value": round(value, 1), "unit": "GB/s", "n_gpus": world,
            "steps": K, "warmup": W, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": cfg["dtype"], "data": "synthetic",
            "config": workload_config(cfg, args.config, B, world),
            "us_per_step": round(ms_per_step * 1e3, 1), "tok_per_s": round(B * world / (ms_per_step * 1e-3), 1),
            "algorithmic_bytes_per_step": step_bytes * world, "per_call": per_call, "roofline": roofline,
            "cpu_baseline": cpu, "cpu_baseline_reference": cpu_ref, "eager_gpu": eager, "e2e": e2e,
            "gpu_launches": launches, "clocks": clocks,
            "tensor_tflops": round(vote_flops / (ms_per_step * 1e-3) / 1e12, 1) if vote_flops else None,
            "rank_cpu_binding": binding, "configs": table, "strong": strong,
            "library": os.path.relpath(_engine.library_path(), ROOT),
        }
        if world > 1:
            line["cpu_baseline_note"] = "cpu_baseline is measured on rank 0 at N=1 only (see the N=1 line)"
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(cfg, B, kv, step_bytes, args, device, world, barrier):
    """The same step with the cache resident in pinned HOST memory, through the public API, host <-> device traffic
    inside the timed region.  Two forms are timed, the faster is reported, the other rides along as `alternative`:

    stored_norms  the host cache is a pinned KVSlabCache: K, V and the [B,H,S] key norms recorded when the rows were
                  appended (they were on the GPU then anyway).  The compress functions called on it read 2 bytes per
                  row for scoring and pull ONLY the kept rows of K and V over PCIe; the compressed cache is written
                  to pinned host tensors.  One launch per call, no copy engine, no staging buffer.
    zero_copy     plain pinned (K, V) lists (no norms): the kernels pull the selection region's K rows for the scan,
                  then the kept rows (round 1's e2e).
    """
    import torch
    import torch.distributed as dist

    import kvcompress
    from kvcompress import KVSlabCache, _planner

    slab = max(1, min(args.e2e_slab, B))
    n_slabs = B // slab
    if n_slabs * slab != B:
        slab, n_slabs = B, 1
    fns = [(kvcompress.get_compress_fn(m), {k: v for k, v in kw.items() if not k.startswith("_")}) for m, kw in cfg["calls"]]
    itemsize = kv[0][0].element_size()
    steps = max(2, min(args.steps, 4))
    S = cfg["S"]

    def timed(step_fn):
        """(job time per step = max over ranks of the barrier-bracketed wall clock, each rank's OWN time per step —
        measured before the closing barrier, so a slow rank shows up as itself instead of as everybody's wait)."""
        step_fn()
        barrier()
        t0 = time.perf_counter()
        own = 0.0
        for _ in range(steps):
            t1 = time.perf_counter()
            step_fn()              # ends with this rank's own stream synchronise
            own += time.perf_counter() - t1
        barrier()
        wall = (time.perf_counter() - t0) / steps
        job, per_rank = wall, [own / steps]
        if world > 1:
            t = torch.tensor([wall, own / steps], device=device, dtype=torch.float64)
            parts = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(parts, t)
            job = max(float(p[0].item()) for p in parts)
            per_rank = [float(p[1].item()) for p in parts]
        return job, per_rank

    # one pinned slab of `slab` streams is reused for every slab of the step (same bytes cross PCIe; content synthetic)
    dev_slice = [(k[:slab], v[:slab]) for k, v in kv]
    host_slab = KVSlabCache.from_legacy_cache(dev_slice, capacity=S, pinned=True)   # append: rows + norms -> host
    torch.cuda.synchronize()

    def sn_step():
        outs = None
        for _ in range(n_slabs):
            outs = [fn(host_slab, **kw) for fn, kw in fns]   # pinned slab in -> pinned (K, V) out, synchronous
        return outs

    probe = sn_step()
    d2h_bytes = n_slabs * sum(k.numel() * itemsize + v.numel() * itemsize
                              for out in probe for (k, v), (k0, _) in zip(out, host_slab)
                              if k.data_ptr() != k0.data_ptr())   # untouched layers are returned as they are
    del probe
    # bytes read over PCIe: per compressed layer the kept rows of K and V (2C rows) + 2 bytes per row of the region
    sn_h2d = 0
    for m, kw in cfg["calls"]:
        for p in plans_for(m, [S] * cfg["L"], kw):
            if p.kind == _planner.GATHER:
                sn_h2d += B * cfg["H"] * (2 * p.out_len * cfg["D"] * itemsize + p.region * itemsize)
    sn_s, sn_ranks = timed(sn_step)

    def sndev_step():
        # fetch-and-compress: the compressed cache lands on the GPU (decode continues there); nothing goes back
        outs = None
        for _ in range(n_slabs):
            outs = [fn(host_slab, output_device=device, **kw) for fn, kw in fns]
        torch.cuda.current_stream().synchronize()
        return outs

    sndev_s, sndev_ranks = timed(sndev_step)

    host_in = host_slab.to_legacy_cache()   # the same pinned rows as plain (K, V) views: no norms travel with them

    def zc_step():
        outs = None
        for _ in range(n_slabs):
            outs = [fn(host_in, **kw) for fn, kw in fns]
        return outs

    zc_h2d = step_bytes - d2h_bytes   # R (scan) + 2C (gather) rows per compressed layer
    zc_s, zc_ranks = timed(zc_step)

    def entry(dt_s, ranks, h2d, how):
        return {"value": round(step_bytes * world / dt_s / 1e9, 2), "unit": "GB/s", "h2d_bytes_per_step": h2d,
                "d2h_bytes_per_step": d2h_bytes, "ms_per_step": round(dt_s * 1e3, 2),
                "per_rank_ms": [round(x * 1e3, 1) for x in ranks], "steps": steps, "how": how}

    common = (f"the host-resident cache is a pinned KVSlabCache ({slab} streams x {n_slabs} slabs per step): K, V and the key "
              f"norms recorded at append time live in page-locked host memory; the public compress functions are called on "
              f"it; over PCIe travel 2 B per row of the selection region (norms) + the kept K/V rows (host->device) and the "
              f"compressed cache (device->host, pinned outputs); wall clock, max over ranks; value = the step's algorithmic "
              f"bytes (same figure as the device-resident run) / that time")
    legs = [
        (sn_s, entry(sn_s, sn_ranks, sn_h2d, "stored_norms: " + common + "; every call synchronises before it returns, as "
                     "the reference's CPU path does (queueing the calls with non_blocking=True and synchronising once per "
                     "step measured the same: 293 vs 296 ms, the link is the limit — profiles/r02_e2e_probe.json)")),
        (zc_s, entry(zc_s, zc_ranks, zc_h2d,
                     "zero_copy: plain pinned host (K, V) lists, no stored norms: the kernels read the selection region's K "
                     "rows for the scan and the kept rows over PCIe and write the compressed cache to pinned host memory "
                     "(round 1's e2e)")),
    ]
    legs.sort(key=lambda x: x[0])
    best = legs[0][1]   # the headline stays host buffers in -> host buffers out
    to_dev = entry(sndev_s, sndev_ranks, sn_h2d,
                   "stored_norms, output_device=cuda (NOT the headline: nothing returns to the host): the pinned slab is "
                   "compressed straight onto the GPU, the kept rows cross PCIe once, host to device")
    to_dev["d2h_bytes_per_step"] = 0
    best["alternatives"] = [l[1] for l in legs[1:]] + [to_dev]
    return best


def run_slab(args):
    """The same calls IN PLACE on a KVSlabCache: per decode step `compress_` (one launch, scores from the stored
    key norms, rows slide down inside the slab) and, at steady state (S = cap + 1), `append` of the next token
    (one launch for all layers).  Reported against the SAME algorithmic bytes as the out-of-place functions
    (SURVEY 8d: "In-place mode is reported against the same figure"), so GB/s above the HBM peak means bytes
    that no longer move."""
    import torch

    import kvcompress
    from kvcompress import KVSlabCache, _engine

    if int(os.environ.get("WORLD_SIZE", "1")) != 1:
        raise SystemExit("--mode slab is a single-GPU measurement")
    torch.cuda.set_device(0)
    device = torch.device("cuda", 0)
    cfg = dict(CONFIGS[args.config])
    if args.seq_len:
        cfg["S"] = args.seq_len
    B = args.batch or cfg["B"]
    S = cfg["S"]
    per_call_bytes = call_bytes(cfg, B)
    kv = make_cache(cfg, B, device, seed=1234)
    dt = kv[0][0].dtype
    slabs, news, steady = [], [], []
    for method, kw in cfg["calls"]:
        slab = KVSlabCache.from_legacy_cache(kv, capacity=S + 8)
        plans = slab.plans_for(method, **kw)
        steady.append(all(p.kind == "keep" or p.out_len == S - 1 for p in plans))
        slabs.append(slab)
        # the next decode token, for the layers the call compresses (skipped layers are left at S rows)
        news.append([(torch.randn(B, cfg["H"], 1, cfg["D"], device=device).to(dt),
                      torch.randn(B, cfg["H"], 1, cfg["D"], device=device).to(dt)) if p.kind != "keep" else None
                     for p in plans])
    del kv
    torch.cuda.synchronize()

    def one_step(events=None):
        for i, ((method, kw), slab) in enumerate(zip(cfg["calls"], slabs)):
            if events is not None:
                events[i][0].record()
            slab.compress_(method, **kw)
            if events is not None:
                events[i][1].record()
            if steady[i]:
                slab.append(news[i])        # the next decode token: back to S rows
            else:
                slab.lengths = [S] * cfg["L"]  # prefill-sized compress: rewind (rows stay valid data)
            if events is not None:
                events[i][2].record()

    for _ in range(max(args.warmup, 3)):
        one_step()
    torch.cuda.synchronize()
    K = args.steps
    ev = [[tuple(torch.cuda.Event(enable_timing=True) for _ in range(3)) for _ in cfg["calls"]] for _ in range(K)]
    sampler = ClockSampler(0)
    sampler.start()
    launches0 = _engine.launch_count()
    t0 = time.perf_counter()
    for s in range(K):
        one_step(ev[s])
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3 / K
    launches = _engine.launch_count() - launches0
    clocks = sampler.stop()
    peak, peak_src = measured_peak()
    per_call = {}
    total_ms = 0.0
    for i, (method, _) in enumerate(cfg["calls"]):
        comp = [x[i][0].elapsed_time(x[i][1]) for x in ev]
        app = [x[i][1].elapsed_time(x[i][2]) for x in ev]
        c_ms, a_ms = statistics.mean(comp), statistics.mean(app)
        total_ms += c_ms + (a_ms if steady[i] else 0.0)
        per_call[method] = {"compress_us_mean": round(c_ms * 1e3, 1), "compress_us_min": round(min(comp) * 1e3, 1),
                            "append_us_mean": round(a_ms * 1e3, 1) if steady[i] else None,
                            "algorithmic_bytes": per_call_bytes[i],
                            "effective_gbs": round(per_call_bytes[i] / (c_ms * 1e-3) / 1e9, 1),
                            "steady_state": steady[i]}
    # the same steady-state step (append + compress_) replayed from a CUDA graph: no per-step host work
    graph_us = {}
    for i, ((method, kw), slab) in enumerate(zip(cfg["calls"], slabs)):
        if not steady[i] or any(n is None for n in news[i]) or len(set(slab.lengths)) != 1:
            continue
        slab.compress_(method, **kw)  # the timed loop leaves the slab one token past its cap
        step = slab.capture_step(method, **kw)
        for _ in range(5):
            step()
        torch.cuda.synchronize()
        n_rep = max(K, 20)
        a, b2 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        a.record()
        for _ in range(n_rep):
            step()
        b2.record()
        torch.cuda.synchronize()
        graph_us[method] = {"device_us_per_step": round(a.elapsed_time(b2) * 1e3 / n_rep, 1),
                            "wall_us_per_step": round((time.perf_counter() - t0) * 1e6 / n_rep, 1)}
    line = {
        "metric": "kv_compress_step_throughput", "mode": "slab_in_place", "value": round(sum(per_call_bytes) / (total_ms * 1e-3) / 1e9, 1),
        "unit": "GB/s (same algorithmic bytes as the out-of-place functions)", "n_gpus": 1, "steps": K,
        "warmup": max(args.warmup, 3), "ms_per_step": round(total_ms, 4), "wall_ms_per_step": round(wall_ms, 4),
        "higher_is_better": True, "dtype": cfg["dtype"], "data": "synthetic",
        "config": workload_config(cfg, args.config, B, 1), "tok_per_s": round(B / (total_ms * 1e-3), 1),
        "per_call": per_call, "graph_replay": graph_us or None, "gpu_launches": launches, "clocks": clocks,
        "peak": peak, "peak_source": peak_src,
    }
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "slab":
        run_slab(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
