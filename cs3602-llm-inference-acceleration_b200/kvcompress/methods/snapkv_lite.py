"""SnapKV-lite: pooled inverted-norm voting + observation window (reference methods/snapkv_lite.py:24-154)."""

from dataclasses import replace
from typing import List, Tuple

import torch

from .. import _engine, _planner
from ..query_window import SnapKVQueryWindow
from ._common import as_layer_list, cached_plans, execute, seq_lens, stored_norms


def snapkv_lite_compress(past_key_values, observation_window: int = 32, keep_size: int = 512,
                         pooling_kernel: int = 5, skip_layers: List[int] = [],
                         **kwargs) -> List[Tuple[torch.Tensor, torch.Tensor]]:
    """Keep the last ``observation_window`` tokens plus the ``keep_size - observation_window`` prefix
    tokens with the highest pooled score ``avg_pool1d(max_norm + 1e-6 - ||K||_2, pooling_kernel)``.

    ``obs_queries=`` (keyword-only extension read from ``**kwargs`` so the drop-in signature is unchanged; off by
    default — the reference has no queries): one ``[B, H*G, W, D]`` tensor per
    layer holding the query states of the last ``W = observation_window`` positions.  The prefix score then
    becomes the SnapKV vote ``softmax(q.K^T / sqrt(D)).sum(window queries, group heads)`` computed on the tensor
    cores, pooled, selected and gathered exactly as above — all in ONE launch (``_engine.snapkv_vote_compress``).
    ``obs_lse=`` (optional, with ``obs_queries``): per layer the ``[B, H*G, W]`` float32 log-sum-exp of those queries'
    attention rows, as returned by a flash-attention forward; the kernel then reads K once instead of twice.
    ``obs_queries`` may also be a :class:`kvcompress.SnapKVQueryWindow` fed by the model's own forwards: its window must
    be ``observation_window`` long and full on every layer that votes (``ValueError`` otherwise)."""
    obs_queries = kwargs.get("obs_queries")
    layers = as_layer_list(past_key_values)
    if not layers:
        return layers
    plans = cached_plans(_planner.plan_snapkv, seq_lens(layers), observation_window, keep_size, pooling_kernel,
                         skip_layers=skip_layers)
    if obs_queries is None:
        return execute(layers, plans, norms=stored_norms(past_key_values),
                   non_blocking=kwargs.get("non_blocking", False), output_device=kwargs.get("output_device"))
    plans, obs_queries = vote_plans(plans, obs_queries, observation_window, len(layers))
    return _engine.snapkv_vote_compress(layers, plans, obs_queries, observation_window, lse=kwargs.get("obs_lse"))


_VOTE_PLANS = {}


def vote_plans(plans, obs_queries, window: int, n_layers: int):
    """The snapkv ``plans`` of a vote (function and ``KVSlabCache.compress_``): every compressed layer ranks its prefix
    by its votes (``SCORE_GIVEN_SCORE``).  Returns ``(PlanSet, per-layer queries)``, a :class:`SnapKVQueryWindow`
    resolved; ``ValueError`` unless there is one entry per layer and every layer that votes has one."""
    voted = [li for li, p in enumerate(plans) if p.kind == _planner.GATHER and p.k_sel > 0]
    if isinstance(obs_queries, SnapKVQueryWindow):
        obs_queries = obs_queries.queries_for(window, voted)
    if len(obs_queries) != n_layers:
        raise ValueError(f"obs_queries: {len(obs_queries)} entries for {n_layers} layers")
    for li in voted:
        if obs_queries[li] is None:
            raise ValueError(f"obs_queries[{li}] is missing for a layer that is compressed")
    # a decode loop votes with the same (cached) plans every step: rewrite them once, not ahead of every vote launch
    hit = _VOTE_PLANS.get(id(plans))
    if hit is None or hit[0] is not plans:
        hit = (plans, _engine.PlanSet([replace(p, score=_planner.SCORE_GIVEN_SCORE) if li in voted else p
                                       for li, p in enumerate(plans)]))
        if len(_VOTE_PLANS) > 64:
            _VOTE_PLANS.clear()
        _VOTE_PLANS[id(plans)] = hit
    return hit[1], obs_queries


__all__ = ["snapkv_lite_compress"]
