"""The SnapKV observation window on the device: the queries of the last W positions of every layer, for the vote.

``snapkv_lite_compress(..., obs_queries=...)`` scores each prefix key by the softmax attention mass it receives from
the queries of the last W positions (the tcgen05 vote of ``csrc/kvc_vote.cuh``).  A decode forward yields one query
per head, so those queries are spread over W forwards.  :class:`SnapKVQueryWindow` keeps them: a ``[B, Hq, W, D]``
buffer per layer, allocated once, that :meth:`SnapKVQueryWindow.push` slides forward by the rows of a forward in ONE
``kvc_query_window_push`` launch for every layer (no ATen kernel, no synchronisation).

    window = kvcompress.SnapKVQueryWindow.for_model(model, batch=1, window=32)
    with torch.inference_mode(), kvcompress.capture_queries(model) as cap:
        out = model(ids, past_key_values=cache, use_cache=True)
    window.push(cap)
    cache.compress_("snapkv_lite", observation_window=32, keep_size=512, obs_queries=window)

Alignment: row i of the window is the query of the position whose key sits at row ``S - W + i`` of the cache.  That
holds when every forward's queries were pushed, in order, and every compaction keeps the last W rows (snapkv_lite's
tail is the observation window).  It is not checked.
"""

from __future__ import annotations

import struct
from typing import List, Optional, Sequence, Union

import torch

from . import _engine
from .capture import QueryCapture

MAX_WINDOW = 128           # the vote stacks G * W query rows into one 128-row MMA tile
VOTE_HEAD_DIMS = (64, 80, 128)


def _fp32(x: float) -> float:
    return struct.unpack("f", struct.pack("f", x))[0]


class SnapKVQueryWindow:
    """Per layer, the post-RoPE queries of the last ``filled[l] <= window`` positions, ``[B, Hq, window, D]`` in
    position order (``queries[l]``, ready for ``obs_queries=``).  16-bit only, as the vote."""

    def __init__(self, num_layers: int, batch: int, num_heads: int, head_dim: int, window: int,
                 dtype: torch.dtype = torch.bfloat16, device: Optional[Union[str, torch.device]] = None):
        if not 1 <= int(window) <= MAX_WINDOW:
            raise ValueError(f"window must be in [1, {MAX_WINDOW}], got {window}")
        if dtype not in (torch.bfloat16, torch.float16):
            raise ValueError(f"the q.K^T vote runs on bfloat16/float16 queries, got {dtype}")
        if num_layers < 1 or batch < 1 or num_heads < 1 or head_dim < 1:
            raise ValueError("num_layers, batch, num_heads and head_dim must be >= 1")
        self.num_layers, self.batch, self.num_heads, self.head_dim = int(num_layers), int(batch), int(num_heads), \
            int(head_dim)
        self.window, self.dtype = int(window), dtype
        self.device = torch.device(device if device is not None else "cuda")
        self._buf = torch.empty((self.num_layers, self.batch, self.num_heads, self.window, self.head_dim), dtype=dtype,
                                device=self.device)
        self.queries: List[torch.Tensor] = list(self._buf.unbind(0))
        self.filled: List[int] = [0] * self.num_layers
        self._reorder_recs: Optional[_engine.RegionRecords] = None   # built by the first reorder

    @classmethod
    def for_model(cls, model, batch: int, window: int) -> "SnapKVQueryWindow":
        """A window shaped for ``model`` (layers, query heads and head_dim from its config; dtype and device from its
        parameters)."""
        cfg = model.config
        head_dim = getattr(cfg, "head_dim", None) or cfg.hidden_size // cfg.num_attention_heads
        p = next(model.parameters())
        return cls(cfg.num_hidden_layers, batch, cfg.num_attention_heads, head_dim, window, p.dtype, p.device)

    def reset(self) -> None:
        """Forget every query (the buffers stay allocated)."""
        self.filled = [0] * self.num_layers

    def push(self, queries: Union[QueryCapture, Sequence[Optional[torch.Tensor]]]) -> "SnapKVQueryWindow":
        """Append a forward's queries: a :class:`QueryCapture` or a per-layer list of ``[B, Hq, T, D]`` tensors
        (``None``: the layer is left as it is).  One launch for every layer that ran.  A capture must have run
        causally (no mask) with the ``head_dim ** -0.5`` scaling the vote uses; otherwise ``ValueError``."""
        if isinstance(queries, QueryCapture):
            want = _fp32(self.head_dim ** -0.5)
            for l, q in enumerate(queries.queries):
                if q is None:
                    continue
                if queries.scaling[l] is None or _fp32(queries.scaling[l]) != want:
                    raise ValueError(f"layer {l}: attention scaling {queries.scaling[l]} is not head_dim ** -0.5; the "
                                     "vote's softmax scale is fixed at 1 / sqrt(head_dim)")
                if queries.masks[l] is not None:
                    raise ValueError(f"layer {l}: the forward ran with an attention mask (padding or a multi-token "
                                     "forward on a non-empty cache); the vote applies the causal rule inside the "
                                     "window only")
            queries = queries.queries
        if len(queries) != self.num_layers:
            raise ValueError(f"{len(queries)} query entries for {self.num_layers} layers")
        recs = [(q, self.queries[l], self.filled[l]) for l, q in enumerate(queries) if q is not None and q.size(2) > 0]
        _engine.query_window_push(recs, self.window)
        for l, q in enumerate(queries):
            if q is not None:
                self.filled[l] = min(self.window, self.filled[l] + q.size(2))
        return self

    def _reorder_records(self, batch: int, device: torch.device) -> bytes:
        """``kvc_batch_region`` records of the filled rows of every layer, for a batch reorder.  The window buffer is
        allocated once, so its pointers and strides are packed once; each call writes the rows from ``filled``."""
        buf = self._buf
        if batch != self.batch or torch.device(device) != buf.device:
            raise ValueError(f"SnapKVQueryWindow of batch {self.batch} on {buf.device}, reordered with a cache of "
                             f"batch {batch} on {device}")
        e = buf.element_size()
        if self._reorder_recs is None:
            self._reorder_recs = _engine.RegionRecords(
                [(buf[l].data_ptr(), buf.stride(1) * e, buf.stride(2) * e, 0, self.num_heads, e)
                 for l in range(self.num_layers)])
        return self._reorder_recs.packed([n * self.head_dim * e for n in self.filled])

    def reorder_(self, index) -> "SnapKVQueryWindow":
        """Beam search's reorder of the window: batch entry b of the filled rows of every layer becomes what entry
        ``index[b]`` held (``index_select(0, index)``), ONE ``kvc_batch_reorder`` launch.  ``index`` as in
        :meth:`KVSlabCache.reorder_`, which takes this window as a follower to move it in the slab's launch."""
        recs = self._reorder_records(self.batch, self._buf.device)
        _engine.batch_reorder(recs, _engine.reorder_index(index, self.batch, self._buf.device), self.batch)
        return self

    def queries_for(self, observation_window: int, layers: Sequence[int]) -> List[torch.Tensor]:
        """``queries`` for a compression whose voted layers are ``layers``: ``ValueError`` unless the window is
        ``observation_window`` long and full on every one of them."""
        if observation_window != self.window:
            raise ValueError(f"observation_window {observation_window} != the query window's {self.window}")
        short = [l for l in layers if self.filled[l] < self.window]
        if short:
            raise ValueError(f"layers {short} hold {[self.filled[l] for l in short]} of the {self.window} window "
                             "queries the vote needs")
        return self.queries


def window_for_harness(model, compress_fn, compress_kwargs: dict, batch: int) -> SnapKVQueryWindow:
    """The observation window of a ``scores="queries"`` harness run, after every check that can fail before the first
    forward: ``compress_fn`` is ``snapkv_lite_compress``, the model is 16-bit, and the vote covers its shape."""
    from .methods import snapkv_lite_compress

    if compress_fn is not snapkv_lite_compress:
        raise ValueError("scores='queries' scores keys with the SnapKV vote: compress_fn must be snapkv_lite_compress "
                         f"(or None), got {getattr(compress_fn, '__name__', compress_fn)}")
    cfg = model.config
    dtype = next(model.parameters()).dtype
    if dtype not in (torch.bfloat16, torch.float16):
        raise ValueError(f"scores='queries': the q.K^T vote runs on bfloat16/float16 models, got {dtype}")
    window = int(compress_kwargs.get("observation_window", 32))
    heads = cfg.num_attention_heads
    group = heads // (getattr(cfg, "num_key_value_heads", None) or heads)
    if group * window > MAX_WINDOW:
        raise ValueError(f"scores='queries': group size {group} x observation_window {window} exceeds the "
                         f"{MAX_WINDOW} query rows of one MMA")
    head_dim = getattr(cfg, "head_dim", None) or cfg.hidden_size // heads
    if head_dim not in VOTE_HEAD_DIMS:
        raise ValueError(f"scores='queries': head_dim {head_dim}; the vote kernel covers head_dim {VOTE_HEAD_DIMS}")
    return SnapKVQueryWindow.for_model(model, batch, window)


__all__ = ["SnapKVQueryWindow"]
