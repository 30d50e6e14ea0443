"""Generation timing with KV-cache compression (reference ``kvcompress/benchmark.py:23-260``).

``measure_generation_metrics`` — prefill, then greedy decode with compression after every step: TTFT, TPOT,
tokens/s.  ``benchmark`` — quality and timing in one pass over ``eval_tokens`` (delegates to
``evaluate_with_compression``, as the reference does :176-215).  ``run_benchmark_suite`` — a list of method
configs.  All take ``cache="dynamic" | "slab"`` (see ``evaluate.py``) and ``input_ids=`` for offline runs.
"""

from __future__ import annotations

import time
from typing import Callable, Dict, List, Optional

import torch

from .evaluate import _check_scores, _forward, evaluate_with_compression, method_name_of, new_slab_for_model
from .query_window import window_for_harness
from .utils import normalize_kv_cache, to_dynamic_cache


def measure_generation_metrics(model, tokenizer=None, text: str = "", compress_fn: Optional[Callable] = None,
                               compress_kwargs: Optional[Dict] = None, max_new_tokens: int = 1000,
                               max_input_tokens: int = 3000, skip_layers: List[int] = [0, 1],
                               device: Optional[torch.device] = None, *, input_ids: Optional[torch.Tensor] = None,
                               cache: str = "dynamic", scores: str = "norms") -> Dict[str, float]:
    """TTFT / TPOT / throughput of greedy generation with compression after the prefill and after every token.
    ``scores="queries"``: snapkv_lite votes with the model's own queries (the prompt's last ``observation_window``
    queries after the prefill, then one more per decode step; see ``evaluate.py``)."""
    _check_scores(scores)
    if device is None:
        device = next(model.parameters()).device
    compress_kwargs = dict(compress_kwargs or {})
    if input_ids is None:
        input_ids = tokenizer.encode(text, return_tensors="pt")
    input_ids = input_ids[:, :max_input_tokens].to(device)
    input_length = input_ids.shape[1]
    eos = getattr(tokenizer, "eos_token_id", None) if tokenizer is not None else None
    window = None
    if scores == "queries" and compress_fn is not None:
        window = window_for_harness(model, compress_fn, compress_kwargs, input_ids.shape[0])
        compress_kwargs["obs_queries"] = window

    slab = method = None
    past_key_values = None
    if cache == "slab":
        method = method_name_of(compress_fn) if compress_fn is not None else None
        if compress_fn is not None and method is None:
            raise ValueError("cache='slab' needs a registered compress function")
        slab = new_slab_for_model(model, input_ids.shape[0], capacity=input_length + max_new_tokens, device=device)
        past_key_values = slab.as_hf_cache()

    def compress(pkv):
        if slab is not None:
            if method is not None:
                slab.compress_(method, skip_layers=skip_layers, **compress_kwargs)
            return pkv
        if compress_fn is None or pkv is None:
            return pkv
        return to_dynamic_cache(compress_fn(list(normalize_kv_cache(pkv)), skip_layers=skip_layers, **compress_kwargs))

    model.eval()
    generated = []
    total_start = time.perf_counter()
    with torch.inference_mode():
        outputs = _forward(model, window, input_ids, past_key_values=past_key_values, use_cache=True, return_dict=True)
        next_token = torch.argmax(outputs.logits[:, -1, :], dim=-1, keepdim=True)
        generated.append(next_token)
        if device.type == "cuda":
            torch.cuda.synchronize(device)
        ttft = time.perf_counter() - total_start
        past_key_values = compress(outputs.past_key_values)
        for _ in range(max_new_tokens - 1):
            outputs = _forward(model, window, next_token, past_key_values=past_key_values, use_cache=True,
                              return_dict=True)
            next_token = torch.argmax(outputs.logits[:, -1, :], dim=-1, keepdim=True)
            generated.append(next_token)
            if eos is not None and next_token.numel() == 1 and next_token.item() == eos:
                break
            past_key_values = compress(outputs.past_key_values)
        if device.type == "cuda":
            torch.cuda.synchronize(device)
    total_time = time.perf_counter() - total_start
    n = len(generated)
    return {"ttft": ttft, "tpot": (total_time - ttft) / max(n - 1, 1), "throughput": n / total_time if total_time else 0.0,
            "total_time": total_time, "num_tokens": n, "input_length": input_length}


def benchmark(model, tokenizer=None, text: str = "", compress_fn: Optional[Callable] = None,
              compress_kwargs: Optional[Dict] = None, max_new_tokens: int = 1000, eval_tokens: int = 3000,
              skip_layers: List[int] = [0, 1], device: Optional[torch.device] = None, **extra) -> Dict[str, float]:
    """Timing and quality in one pass over ``eval_tokens`` (reference benchmark.py:145-215)."""
    m = evaluate_with_compression(model=model, tokenizer=tokenizer, text=text, compress_fn=compress_fn,
                                  compress_kwargs=compress_kwargs or {}, max_tokens=eval_tokens, skip_layers=skip_layers,
                                  device=device, show_progress=extra.pop("show_progress", True), **extra)
    return {"ttft": m["ttft"], "tpot": m["tpot"], "throughput": m["throughput"], "total_time": m["total_time"],
            "perplexity": m["perplexity"], "accuracy": m["accuracy"], "eval_tokens": m["num_tokens"],
            "final_cache_size": m["final_cache_size"]}


def run_benchmark_suite(model, tokenizer=None, text: str = "", methods_config: List[Dict] = (), max_new_tokens: int = 1000,
                        eval_tokens: int = 3000, skip_layers: List[int] = [0, 1],
                        device: Optional[torch.device] = None, **extra) -> List[Dict[str, float]]:
    """One ``benchmark`` per ``{"name", "compress_fn", "kwargs"}`` entry (reference benchmark.py:218-290)."""
    results = []
    for config in methods_config:
        res = benchmark(model, tokenizer, text, compress_fn=config.get("compress_fn"), compress_kwargs=config.get("kwargs", {}),
                        max_new_tokens=max_new_tokens, eval_tokens=eval_tokens, skip_layers=skip_layers, device=device,
                        **extra)
        res["name"] = res["method"] = config.get("name", "unknown")
        results.append(res)
    return results


def print_benchmark_summary(results: List[Dict[str, float]]) -> None:
    """Table of ``run_benchmark_suite`` results and each method's change against the baseline row (the entry named
    "baseline", else the first) — reference benchmark.py:293-350."""
    cols = (("ttft", "TTFT(s)", "{:>10.4f}"), ("tpot", "TPOT(s)", "{:>10.4f}"), ("throughput", "Thruput", "{:>10.2f}"),
            ("perplexity", "PPL", "{:>10.2f}"), ("accuracy", "Acc", "{:>10.2%}"), ("final_cache_size", "Cache", "{:>8}"))
    rule = "=" * 90
    print("\n" + rule + "\nBENCHMARK SUMMARY\n" + rule)
    print(f"{'Method':<20} " + " ".join(f"{title:>{8 if key == 'final_cache_size' else 10}}" for key, title, _ in cols))
    print("-" * 90)
    label = lambda r: str(r.get("method", r.get("name", "unknown")))
    for r in results:
        print(f"{label(r)[:20]:<20} " + " ".join(fmt.format(r[key]) for key, _, fmt in cols))
    print(rule)
    base = next((r for r in results if label(r) == "baseline"), results[0] if results else None)
    if base is None or len(results) < 2:
        return
    print("\nAgainst " + label(base) + " (throughput: higher is better; TPOT, PPL: lower is better):")
    for r in results:
        if r is base:
            continue
        thr = (r["throughput"] / base["throughput"] - 1) * 100 if base["throughput"] > 0 else 0.0
        tpot = (1 - r["tpot"] / base["tpot"]) * 100 if base["tpot"] > 0 else 0.0
        ppl = (r["perplexity"] / base["perplexity"] - 1) * 100 if base["perplexity"] > 0 else 0.0
        print(f"  {label(r)[:20]:<20} throughput {thr:+.1f}%   TPOT {tpot:+.1f}% faster   PPL {ppl:+.1f}%")


__all__ = ["measure_generation_metrics", "benchmark", "run_benchmark_suite", "print_benchmark_summary"]
