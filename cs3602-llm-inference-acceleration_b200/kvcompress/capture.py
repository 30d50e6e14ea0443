"""Record the post-RoPE queries and cached keys of a transformers model's attention layers.

``H2OScoreSlab.update_from_queries`` rebuilds the attention probabilities on the device from the queries and keys, so
the model need not return them (``output_attentions=True`` needs ``attn_implementation="eager"`` and materialises
``[B, Hq, T, key_len]`` per layer).  :func:`capture_queries` switches a model to an attention function registered as
``"kvcompress_sdpa"``: it records its arguments per layer and returns ``sdpa_attention_forward(...)`` unchanged, so
the model computes what it computes under ``attn_implementation="sdpa"``.

    with torch.inference_mode(), kvcompress.capture_queries(model) as cap:
        out = model(ids, past_key_values=cache, use_cache=True)
    manager.update_from_queries(cap.queries, cap.keys, cap.masks, cap.scaling)

The records are the tensors the attention layers saw: the queries, the keys as the cache returned them (a view of a
slab cache, un-repeated ``[B, Hkv, key_len, D]``) and the mask (``None`` when the layer ran causally).  They are valid
until the cache is next appended to or compacted.  transformers is imported on first use.
"""

from __future__ import annotations

import contextlib
from typing import List, Optional

import torch

ATTN_NAME = "kvcompress_sdpa"

_registered = False
_active: List["QueryCapture"] = []


class QueryCapture:
    """Per-layer records of the last forward under :func:`capture_queries` (``None`` for a layer that did not run):
    ``queries[l]`` ``[B, Hq, T, D]``, ``keys[l]`` ``[B, Hkv, key_len, D]``, ``masks[l]`` a bool ``[B, 1, T, key_len]``
    mask (True = visible) or ``None`` (causal), ``scaling[l]`` the logit scale."""

    def __init__(self, num_layers: int):
        self.num_layers = num_layers
        self.clear()

    def clear(self) -> None:
        self.queries: List[Optional[torch.Tensor]] = [None] * self.num_layers
        self.keys: List[Optional[torch.Tensor]] = [None] * self.num_layers
        self.masks: List[Optional[torch.Tensor]] = [None] * self.num_layers
        self.scaling: List[Optional[float]] = [None] * self.num_layers

    def _record(self, layer_idx: int, query, key, mask, scaling: float) -> None:
        if layer_idx >= self.num_layers:
            grow = layer_idx + 1 - self.num_layers
            for lst in (self.queries, self.keys, self.masks, self.scaling):
                lst.extend([None] * grow)
            self.num_layers = layer_idx + 1
        self.queries[layer_idx] = query
        self.keys[layer_idx] = key
        self.masks[layer_idx] = mask
        self.scaling[layer_idx] = scaling


def _capture_attention(module, query, key, value, attention_mask, dropout: float = 0.0, scaling=None, **kwargs):
    """``sdpa_attention_forward`` that first records its arguments into the active :class:`QueryCapture`."""
    from transformers.integrations.sdpa_attention import sdpa_attention_forward

    if _active:
        if kwargs.get("softcap") is not None:
            raise ValueError("capture_queries: logit soft-capping changes the probabilities; it is not reproduced")
        if kwargs.get("s_aux") is not None or kwargs.get("sinks") is not None:
            raise ValueError("capture_queries: attention sinks change the probabilities; they are not reproduced")
        if dropout and dropout > 0:
            raise ValueError("capture_queries: attention dropout > 0 (training mode) is not reproduced")
        if attention_mask is not None and attention_mask.dtype != torch.bool:
            raise ValueError(f"capture_queries: a {attention_mask.dtype} attention mask is not supported (bool only)")
        layer_idx = getattr(module, "layer_idx", None)
        if layer_idx is None:
            raise ValueError("capture_queries: the attention module has no layer_idx")
        s = float(scaling) if scaling is not None else query.size(-1) ** -0.5
        _active[-1]._record(int(layer_idx), query, key, attention_mask, s)
    return sdpa_attention_forward(module, query, key, value, attention_mask, dropout=dropout, scaling=scaling, **kwargs)


def _register() -> None:
    global _registered
    if _registered:
        return
    from transformers import AttentionInterface, AttentionMaskInterface
    from transformers.masking_utils import sdpa_mask

    AttentionInterface.register(ATTN_NAME, _capture_attention)
    AttentionMaskInterface.register(ATTN_NAME, sdpa_mask)
    _registered = True


@contextlib.contextmanager
def capture_queries(model):
    """Run ``model`` on the recording SDPA attention inside the context; yields the :class:`QueryCapture` that the
    forwards fill.  The model's attention implementation is restored on exit, exceptions included."""
    _register()
    prev = model.config._attn_implementation
    cap = QueryCapture(getattr(model.config, "num_hidden_layers", 0) or 0)
    model.set_attn_implementation(ATTN_NAME)
    _active.append(cap)
    try:
        yield cap
    finally:
        _active.remove(cap)
        model.set_attn_implementation(prev)


__all__ = ["capture_queries", "QueryCapture"]
