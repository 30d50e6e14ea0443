"""Token-by-token evaluation with KV-cache compression — the caller loop on both sides of the hot path.

Same entry point, arguments and result keys as the reference's ``kvcompress/evaluate.py:26-226``
(``evaluate_with_compression``): one token per forward pass, compression after EVERY pass, per-token NLL
with ``CrossEntropyLoss(reduction="none")``, PPL = exp(mean NLL), TTFT/TPOT over all tokens.

Two cache paths run the identical loop:

``cache="dynamic"``  the reference's shape (evaluate.py:150-166): the model's ``DynamicCache`` is flattened
                     with ``normalize_kv_cache``, compressed by ``compress_fn`` (fresh tensors) and rebuilt with
                     ``to_dynamic_cache`` — every step re-allocates and copies the cache twice;
``cache="slab"``     a :class:`KVSlabCache` is the model's cache object: HF's ``update`` appends in place, and
                     ``compress_`` compacts every layer in place in one launch (SURVEY.md §8f rank 1).

Two score sources for ``snapkv_lite_compress``:

``scores="norms"``   the reference's SnapKV-lite: prefix keys ranked by pooled inverted key norms;
``scores="queries"`` SnapKV proper: every forward runs under :func:`kvcompress.capture_queries`, a
                     :class:`SnapKVQueryWindow` keeps each layer's queries of the last ``observation_window``
                     positions on the device, and the prefix keys are ranked by the attention mass those queries give
                     them (the tcgen05 vote, ``obs_queries=window``).  16-bit models, ``compress_fn`` snapkv_lite or
                     ``None``, ``G * observation_window <= 128``.

``tokenizer`` only needs ``encode(text, return_tensors="pt")``; pass ``input_ids=`` to skip it (offline runs).
"""

from __future__ import annotations

import math
import time
from typing import Callable, Dict, List, Optional

import torch
from torch.nn import CrossEntropyLoss

from .capture import capture_queries
from .query_window import window_for_harness
from .slab_cache import KVSlabCache
from .utils import normalize_kv_cache, to_dynamic_cache

_EMPTY = {"perplexity": float("inf"), "accuracy": 0.0, "num_tokens": 0, "final_cache_size": 0, "ttft": 0.0,
          "tpot": 0.0, "throughput": 0.0, "total_time": 0.0}


def method_name_of(compress_fn: Callable) -> Optional[str]:
    """Registry name of a compress function (the in-place path is addressed by name)."""
    from .methods import COMPRESS_METHODS

    for name, fn in COMPRESS_METHODS.items():
        if fn is compress_fn:
            return name
    return None


def new_slab_for_model(model, batch: int, capacity: int, dtype=None, device=None) -> KVSlabCache:
    """A slab cache shaped for ``model`` (KV heads and head_dim from its config)."""
    cfg = model.config
    heads = getattr(cfg, "num_key_value_heads", None) or cfg.num_attention_heads
    head_dim = getattr(cfg, "head_dim", None) or cfg.hidden_size // cfg.num_attention_heads
    p = next(model.parameters())
    return KVSlabCache(cfg.num_hidden_layers, batch, heads, head_dim, capacity, dtype or p.dtype, device or p.device)


def _check_scores(scores: str) -> None:
    if scores not in ("norms", "queries"):
        raise ValueError(f"scores must be 'norms' or 'queries', got {scores!r}")


def _forward(model, window, *args, **kwargs):
    """``model(*args, **kwargs)``; with a query window, under :func:`capture_queries`, the queries pushed after."""
    if window is None:
        return model(*args, **kwargs)
    with capture_queries(model) as capture:
        outputs = model(*args, **kwargs)
    window.push(capture)
    return outputs


def _final_cache_size(lengths: List[int], skip_layers) -> int:
    for layer_idx, n in enumerate(lengths):  # a layer that is actually compressed (reference :205-216)
        if layer_idx not in skip_layers:
            return n
    return lengths[0] if lengths else 0


def evaluate_with_compression(model, tokenizer=None, text: str = "", compress_fn: Optional[Callable] = None,
                              compress_kwargs: Optional[Dict] = None, max_tokens: int = 3000,
                              skip_layers: List[int] = [0, 1], device: Optional[torch.device] = None,
                              show_progress: bool = True, *, input_ids: Optional[torch.Tensor] = None,
                              cache: str = "dynamic", return_nlls: bool = False,
                              scores: str = "norms") -> Dict[str, float]:
    """PPL / accuracy / TTFT / TPOT with ``compress_fn`` applied after every token (reference evaluate.py:26-226).
    ``scores="queries"``: snapkv_lite votes with the model's own queries (module docstring)."""
    if cache not in ("dynamic", "slab"):
        raise ValueError(f"cache must be 'dynamic' or 'slab', got {cache!r}")
    _check_scores(scores)
    if device is None:
        device = next(model.parameters()).device
    compress_kwargs = dict(compress_kwargs or {})
    if input_ids is None:
        input_ids = tokenizer.encode(text, return_tensors="pt")
    input_ids = input_ids[:, :max_tokens].to(device)
    seq_len = input_ids.shape[1]
    window = None
    if scores == "queries" and compress_fn is not None:
        window = window_for_harness(model, compress_fn, compress_kwargs, input_ids.shape[0])
        compress_kwargs["obs_queries"] = window
    if seq_len < 2:
        return dict(_EMPTY)

    slab = hf_cache = method = None
    if cache == "slab":
        if compress_fn is not None:
            method = method_name_of(compress_fn)
            if method is None or method == "h2o_attention":
                raise ValueError("cache='slab' needs a registered compress function with an in-place form")
        slab = new_slab_for_model(model, input_ids.shape[0], capacity=seq_len, device=device)
        hf_cache = slab.as_hf_cache()

    loss_fn = CrossEntropyLoss(reduction="none")
    past_key_values = hf_cache
    nlls_dev, correct_dev, token_times = [], [], []
    ttft = None
    steps = range(seq_len - 1)
    if show_progress:
        try:
            from tqdm import tqdm

            steps = tqdm(steps, desc="Evaluating")
        except Exception:
            pass
    model.eval()
    vocab = model.config.vocab_size
    total_start = time.perf_counter()
    with torch.inference_mode():
        for idx in steps:
            token_start = time.perf_counter()
            outputs = _forward(model, window, input_ids[:, idx:idx + 1], past_key_values=past_key_values,
                              use_cache=True)
            logits = outputs.logits[:, -1, :].view(-1, vocab)
            target = input_ids[:, idx + 1:idx + 2].view(-1)
            nll = loss_fn(logits, target)
            # the reference reads nll.item() here (:139), a per-token host sync; keep that contract
            nlls_dev.append(float(nll.mean().item()))
            correct_dev.append(float((torch.argmax(logits, dim=-1) == target).float().mean().item()))
            if slab is not None:
                if method is not None:
                    slab.compress_(method, skip_layers=skip_layers, **compress_kwargs)
            else:
                past_key_values = outputs.past_key_values
                if compress_fn is not None and past_key_values is not None:
                    kv_list = list(normalize_kv_cache(past_key_values))
                    past_key_values = to_dynamic_cache(compress_fn(kv_list, skip_layers=skip_layers, **compress_kwargs))
            token_time = time.perf_counter() - token_start
            token_times.append(token_time)
            if ttft is None:
                ttft = token_time
    total_time = time.perf_counter() - total_start

    num_tokens = len(nlls_dev)
    tpot = sum(token_times[1:]) / (num_tokens - 1) if num_tokens > 1 else (ttft or 0.0)
    if slab is not None:
        lengths = list(slab.lengths)
    elif past_key_values is not None:
        lengths = [k.size(2) for k, _ in normalize_kv_cache(past_key_values)]
    else:
        lengths = []
    result = {
        "perplexity": math.exp(sum(nlls_dev) / num_tokens),
        "accuracy": sum(correct_dev) / num_tokens,
        "num_tokens": num_tokens,
        "final_cache_size": _final_cache_size(lengths, skip_layers),
        "ttft": ttft or 0.0,
        "tpot": tpot,
        "throughput": num_tokens / total_time if total_time > 0 else 0.0,
        "total_time": total_time,
    }
    if return_nlls:
        result["nlls"] = nlls_dev
        result["cache_lengths"] = lengths
    return result


def evaluate_baseline(model, tokenizer=None, text: str = "", max_tokens: int = 3000,
                      device: Optional[torch.device] = None, show_progress: bool = False, **extra) -> Dict[str, float]:
    """The same loop with no compression (reference evaluate.py:229-259)."""
    return evaluate_with_compression(model=model, tokenizer=tokenizer, text=text, compress_fn=None, max_tokens=max_tokens,
                                     device=device, show_progress=show_progress, **extra)


def compare_methods(model, tokenizer=None, text: str = "", methods_config: List[Dict] = (), max_tokens: int = 3000,
                    skip_layers: List[int] = [0, 1], device: Optional[torch.device] = None, **extra) -> List[Dict[str, float]]:
    """One evaluation per ``{"name", "compress_fn", "kwargs"}`` entry; every result carries ``method`` and ``config``
    (reference evaluate.py:262-323)."""
    results = []
    for entry in methods_config:
        label, kwargs = entry.get("name", "unknown"), entry.get("kwargs", {})
        print(f"\nEvaluating {label}...")
        res = evaluate_with_compression(model=model, tokenizer=tokenizer, text=text, compress_fn=entry.get("compress_fn"),
                                        compress_kwargs=kwargs, max_tokens=max_tokens, skip_layers=skip_layers,
                                        device=device, show_progress=extra.pop("show_progress", True), **extra)
        res["method"], res["config"] = label, kwargs
        results.append(res)
        print(f"  PPL: {res['perplexity']:.2f}\n  Accuracy: {res['accuracy']:.2%}\n  Final cache size: {res['final_cache_size']}")
    return results


__all__ = ["evaluate_with_compression", "evaluate_baseline", "compare_methods", "new_slab_for_model", "method_name_of"]
