"""Token-by-token evaluation with attention-score H2O eviction — the caller loop of ``h2o_attention_compress``.

Same entry points, arguments and result keys as the reference's ``kvcompress/evaluate_attention.py:24-330``: every
forward pass runs with ``output_attentions=True``, the :class:`H2OAttentionManager` accumulates the attention mass
each cached position receives, and once the cache exceeds ``start_size + heavy_hitter_size + recent_size`` rows it is
compacted to sinks + heavy hitters + recent rows (the gather runs on the sm_100a kernels with the manager's rows as
``KVC_SCORE_GIVEN_INDEX``), after which the manager starts over — positions have moved (reference :164-177).

``cache="slab"`` runs the same loop on a :class:`KVSlabCache` (the model appends in place, ``compress_`` compacts in
place), as ``evaluate_with_compression`` does.  With an :class:`H2OScoreSlab` as ``h2o_manager`` the score bookkeeping
runs on the device as well: one accumulate launch per update, one compaction launch per compression.

``scores="attentions"`` (the default) needs a model that returns attention weights (``attn_implementation="eager"``).
``scores="queries"`` runs every forward under :func:`kvcompress.capture_queries` (SDPA, no ``output_attentions``) and
updates an :class:`H2OScoreSlab` (the default manager then) from the recorded queries and keys: the probabilities are
rebuilt on the device from fp32 logits.  ``tokenizer`` only needs ``encode(text, return_tensors="pt")`` — pass
``input_ids=`` to skip it (offline runs).

Two semantics of the scores across a compression:

* ``carry_scores=False`` (the default, the reference's reset): after every compression the manager starts over, so
  at steady state (a compression per token) the heavy hitters are ranked by the current token's attention alone;
* ``carry_scores=True`` (cumulative H2O): an ``H2OScoreSlab(carry_scores=True)`` moves its accumulators with the kept
  rows inside the compaction launch; the loop updates the manager once per forward, compresses without handing the
  scores over a second time and never resets, so keys are ranked by the decayed attention of the whole generation.
"""

from __future__ import annotations

import math
import time
from typing import Dict, List, Optional

import torch
from torch.nn import CrossEntropyLoss

from .evaluate import _EMPTY, _final_cache_size, evaluate_with_compression, new_slab_for_model
from .capture import capture_queries
from .methods.h2o_attention import (H2OAttentionManager, H2OScoreSlab, check_carry, h2o_attention_compress,
                                    update_manager)
from .utils import normalize_kv_cache, to_dynamic_cache


def evaluate_with_attention_compression(model, tokenizer=None, text: str = "",
                                        h2o_manager: Optional[H2OAttentionManager] = None, start_size: int = 4,
                                        heavy_hitter_size: int = 64, recent_size: int = 444, max_tokens: int = 3000,
                                        skip_layers: List[int] = [0, 1], device: Optional[torch.device] = None,
                                        show_progress: bool = True, *, input_ids: Optional[torch.Tensor] = None,
                                        cache: str = "dynamic", return_nlls: bool = False,
                                        scores: str = "attentions", carry_scores: bool = False) -> Dict[str, float]:
    """PPL / accuracy / TTFT / TPOT with attention-score H2O applied after every token.  ``h2o_manager``: an
    :class:`H2OAttentionManager` (the default) or an :class:`H2OScoreSlab`; ``cache``: ``"dynamic"`` or ``"slab"``;
    ``scores``: ``"attentions"`` (``output_attentions=True``) or ``"queries"`` (:func:`kvcompress.capture_queries`, an
    :class:`H2OScoreSlab` manager); ``carry_scores``: cumulative scores (an ``H2OScoreSlab(carry_scores=True)``, the
    default manager then) instead of the reference's reset after every compression."""
    if cache not in ("dynamic", "slab"):
        raise ValueError(f"cache must be 'dynamic' or 'slab', got {cache!r}")
    if scores not in ("attentions", "queries"):
        raise ValueError(f"scores must be 'attentions' or 'queries', got {scores!r}")
    if device is None:
        device = next(model.parameters()).device
    if h2o_manager is None:
        manager_cls = H2OScoreSlab if scores == "queries" or carry_scores else H2OAttentionManager
        extra = dict(carry_scores=True) if carry_scores else {}
        h2o_manager = manager_cls(start_size=start_size, heavy_hitter_size=heavy_hitter_size, recent_size=recent_size,
                                  num_layers=getattr(model.config, "num_hidden_layers", 32),
                                  num_heads=getattr(model.config, "num_attention_heads", 32), device=device, **extra)
    else:
        if scores == "queries" and not isinstance(h2o_manager, H2OScoreSlab):
            raise ValueError("scores='queries' needs an H2OScoreSlab manager")
        if carry_scores:
            check_carry(h2o_manager, True)
        h2o_manager.reset()
    use_queries = scores == "queries"
    if input_ids is None:
        input_ids = tokenizer.encode(text, return_tensors="pt")
    input_ids = input_ids[:, :max_tokens].to(device)
    seq_len = input_ids.shape[1]
    if seq_len < 2:
        return dict(_EMPTY)

    budget = start_size + heavy_hitter_size + recent_size
    loss_fn = CrossEntropyLoss(reduction="none")
    past_key_values = slab = None
    if cache == "slab":
        slab = new_slab_for_model(model, input_ids.shape[0], capacity=seq_len, device=device)
        past_key_values = slab.as_hf_cache()
    nlls, correct, token_times = [], [], []
    ttft = None
    steps = range(seq_len - 1)
    if show_progress:
        try:
            from tqdm import tqdm

            steps = tqdm(steps, desc="H2O-Attention Eval")
        except Exception:
            pass
    model.eval()
    vocab = model.config.vocab_size
    total_start = time.perf_counter()
    with torch.inference_mode():
        for idx in steps:
            token_start = time.perf_counter()
            if use_queries:
                with capture_queries(model) as capture:
                    outputs = model(input_ids[:, idx:idx + 1], past_key_values=past_key_values, use_cache=True)
                inputs = dict(attention_queries=capture)
            else:
                outputs = model(input_ids[:, idx:idx + 1], past_key_values=past_key_values, use_cache=True,
                                output_attentions=True)
                inputs = dict(attention_scores=outputs.attentions)
            # cumulative scores: updated once per forward below, the compaction carries the accumulators
            scored = {} if carry_scores else inputs
            logits = outputs.logits[:, -1, :].view(-1, vocab)
            target = input_ids[:, idx + 1:idx + 2].view(-1)
            nlls.append(float(loss_fn(logits, target).mean().item()))
            correct.append(float((torch.argmax(logits, dim=-1) == target).float().mean().item()))

            if slab is not None:
                update_manager(h2o_manager, skip_layers=skip_layers, **inputs)
                if slab.lengths[0] > budget:
                    slab.compress_("h2o_attention", h2o_manager=h2o_manager, start_size=start_size,
                                   heavy_hitter_size=heavy_hitter_size, recent_size=recent_size,
                                   skip_layers=skip_layers, **scored)
                    if not carry_scores:
                        h2o_manager.reset()
            else:
                past_key_values = outputs.past_key_values
                update_manager(h2o_manager, skip_layers=skip_layers, **inputs)
                if past_key_values is not None:
                    kv_list = list(normalize_kv_cache(past_key_values))
                    if kv_list and kv_list[0][0].size(2) > budget:
                        kept = h2o_attention_compress(kv_list, h2o_manager=h2o_manager, start_size=start_size,
                                                      heavy_hitter_size=heavy_hitter_size, recent_size=recent_size,
                                                      skip_layers=skip_layers, **scored)
                        past_key_values = to_dynamic_cache(kept)
                        if not carry_scores:
                            h2o_manager.reset()
            token_time = time.perf_counter() - token_start
            token_times.append(token_time)
            if ttft is None:
                ttft = token_time
    total_time = time.perf_counter() - total_start

    num_tokens = len(nlls)
    if slab is not None:
        lengths = list(slab.lengths)
    else:
        lengths = [k.size(2) for k, _ in normalize_kv_cache(past_key_values)] if past_key_values is not None else []
    result = {
        "perplexity": math.exp(sum(nlls) / num_tokens),
        "accuracy": sum(correct) / num_tokens,
        "num_tokens": num_tokens,
        "final_cache_size": _final_cache_size(lengths, skip_layers),
        "ttft": ttft or 0.0,
        "tpot": sum(token_times[1:]) / (num_tokens - 1) if num_tokens > 1 else (ttft or 0.0),
        "throughput": num_tokens / total_time if total_time > 0 else 0.0,
        "total_time": total_time,
    }
    if return_nlls:
        result["nlls"] = nlls
        result["cache_lengths"] = lengths
    return result


def compare_h2o_methods(model, tokenizer=None, text: str = "", max_tokens: int = 2000,
                        heavy_hitter_sizes: List[int] = [32, 64, 128], skip_layers: List[int] = [0, 1],
                        device: Optional[torch.device] = None, **extra) -> List[Dict]:
    """Baseline, then for every heavy-hitter size (cache budget 512) H2O by key norm and H2O by attention score;
    each result carries ``method`` (reference evaluate_attention.py:231-330)."""
    from .methods import h2o_l2_compress

    if device is None:
        device = next(model.parameters()).device

    def report(label, res):
        res["method"] = label
        print(f"  {label}: PPL {res['perplexity']:.2f}, Acc {res['accuracy']:.2%}, cache {res['final_cache_size']}")
        return res

    results = [report("baseline", evaluate_with_compression(model, tokenizer, text, compress_fn=None,
                                                            max_tokens=max_tokens, device=device, **extra))]
    for hh in heavy_hitter_sizes:
        recent = 512 - 4 - hh
        results.append(report(f"h2o_l2_hh{hh}", evaluate_with_compression(
            model, tokenizer, text, compress_fn=h2o_l2_compress,
            compress_kwargs={"start_size": 4, "heavy_hitter_size": hh, "recent_size": recent},
            max_tokens=max_tokens, skip_layers=skip_layers, device=device, **extra)))
        results.append(report(f"h2o_attn_hh{hh}", evaluate_with_attention_compression(
            model, tokenizer, text, start_size=4, heavy_hitter_size=hh, recent_size=recent, max_tokens=max_tokens,
            skip_layers=skip_layers, device=device, **extra)))
    return results


__all__ = ["evaluate_with_attention_compression", "compare_h2o_methods"]
