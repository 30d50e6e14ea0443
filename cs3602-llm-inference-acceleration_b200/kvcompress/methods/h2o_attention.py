"""H2O with real attention scores (reference methods/h2o_attention.py:28-391).

SURVEY.md §8f lists this as a *next* row: it needs ``output_attentions=True`` model outputs, which
are outside the compress hot path.  It is provided so that every name in ``list_methods()``
resolves and behaves as in the reference:

* without a manager the reference falls back to exactly the ``h2o_l2`` selection
  (h2o_attention.py:337-351) — that runs on the fused sm_100a kernel;
* with a manager, the manager's head-summed top-k indices (shared by every batch entry and head,
  h2o_attention.py:194-213, :318-331) are handed to the gather kernel as caller-supplied indices.

Two managers keep the score bookkeeping:

* `H2OAttentionManager` mirrors the reference's object model in torch arithmetic (CPU or GPU tensors, batch 1);
* `H2OScoreSlab` keeps the decayed accumulators and the head-summed score rows in preallocated device buffers:
  one ``kvc_h2o_accumulate`` launch per update for every layer, and the compaction ranks the rows from the score
  row itself (``KVC_SCORE_GIVEN_SCORE_SHARED``) — no ATen kernel and no host synchronisation on the decode path,
  and every batch entry gets its own heavy hitters.

Two semantics of the accumulators across a compaction:

* reset (the reference's, and the default): the caller resets the manager after every compression, so the heavy
  hitters are ranked by the attention received since the last compaction — at steady state, by one token's attention;
* cumulative (``H2OScoreSlab(carry_scores=True)``): the compaction moves every accumulator row with its token, in the
  same launch (``kvc_*_carry``), and the caller never resets — keys are ranked by the decayed attention they have
  received over the whole generation.
"""

from collections.abc import Mapping
from functools import partial
from typing import Dict, List, Optional, Tuple

import torch

from .. import _engine, _planner
from ._common import as_layer_list, cached_plans, seq_lens
from .h2o_l2 import h2o_l2_compress


def _evenly_spaced(seq_len: int, start_size: int, heavy_hitter_size: int, recent_size: int) -> range:
    """The heavy hitters of a layer without data since the last reset: evenly spaced rows of the middle region,
    relative to it (reference h2o_attention.py:167-177)."""
    middle_len = (seq_len - recent_size) - start_size
    if middle_len <= 0:
        return range(0)
    return range(0, middle_len, max(1, middle_len // heavy_hitter_size))[:heavy_hitter_size]


class H2OAttentionManager:
    """Decayed running sum of attention mass per key position (reference h2o_attention.py:28-213)."""

    def __init__(self, start_size: int = 4, heavy_hitter_size: int = 64, recent_size: int = 444,
                 num_layers: int = 32, num_heads: int = 32, decay_factor: float = 0.9, device=None):
        self.start_size = start_size
        self.heavy_hitter_size = heavy_hitter_size
        self.recent_size = recent_size
        self.total_cache_size = start_size + heavy_hitter_size + recent_size
        self.num_layers = num_layers
        self.num_heads = num_heads
        self.decay_factor = decay_factor
        self.device = device
        self.accumulated_attention: Dict[int, torch.Tensor] = {}
        self.token_positions: Dict[int, torch.Tensor] = {}
        self.current_seq_len = 0

    def reset(self) -> None:
        self.accumulated_attention = {}
        self.token_positions = {}
        self.current_seq_len = 0

    def update_attention_scores(self, attentions, skip_layers: List[int] = []) -> None:
        """acc <- decay * acc (zero-extended, or reset if the cache shrank) + attn.sum(query dim)  (:78-151)."""
        if attentions is None:
            return
        for layer_idx, attn in enumerate(attentions):
            if layer_idx in skip_layers or attn is None:
                continue
            batch, heads, _, key_len = attn.shape
            mass = attn.sum(dim=2)
            prev = self.accumulated_attention.get(layer_idx)
            if prev is None or prev.size(-1) > key_len:
                acc = torch.zeros(batch, heads, key_len, device=attn.device, dtype=attn.dtype)
            else:
                acc = prev * self.decay_factor
                if prev.size(-1) < key_len:
                    grow = torch.zeros(batch, heads, key_len - prev.size(-1), device=attn.device, dtype=attn.dtype)
                    acc = torch.cat([acc, grow], dim=-1)
            self.accumulated_attention[layer_idx] = acc + mass
            self.current_seq_len = key_len

    def get_heavy_hitter_indices(self, layer_idx: int, seq_len: int) -> torch.Tensor:
        """Indices (relative to the middle region, ascending) of its heaviest tokens  (:153-213)."""
        acc = self.accumulated_attention.get(layer_idx)
        if acc is None:
            rows = _evenly_spaced(seq_len, self.start_size, self.heavy_hitter_size, self.recent_size)
            return torch.arange(rows.start, rows.stop, rows.step)
        middle_end = min(seq_len, acc.size(-1)) - self.recent_size
        if middle_end <= self.start_size:
            return torch.tensor([], dtype=torch.long, device=acc.device)
        per_token = acc[:, :, self.start_size:middle_end].sum(dim=1)
        if acc.size(0) == 1:
            per_token = per_token.squeeze(0)
        k = min(self.heavy_hitter_size, middle_end - self.start_size)
        _, top = torch.topk(per_token, k, dim=-1)
        top, _ = torch.sort(top, dim=-1)
        return top

    def compress_plans(self, plans, start_size: int, heavy_hitter_size: int, recent_size: int, batch: int, heads: int,
                       dtype: torch.dtype, device):
        """:meth:`H2OScoreSlab.compress_plans` for this manager (reference h2o_attention.py:318-331): the head-summed
        top-k rows of each compressed layer become caller-supplied rows (``SCORE_GIVEN_INDEX``).  Returns
        ``(plans, {layer: int32 [batch, heads, count] ascending absolute rows on device}, None)``."""
        new_plans = list(plans)  # the manager rewrites per-layer plans below: never touch the cached set
        given = {}
        for li, plan in enumerate(plans):
            if plan.kind != _planner.GATHER or plan.region == 0:
                continue
            middle_len = plan.sel_hi - plan.sel_lo
            picked = self.get_heavy_hitter_indices(li, plan.seq_len)
            count = min(len(picked), heavy_hitter_size, middle_len)  # :321
            if count > 0 and picked.dim() != 1:
                raise ValueError("h2o_attention: the manager's indices are shared across the batch; batch > 1 "
                                 "is not supported (the reference fails on it as well)")
            rows = picked[:count].clamp(0, middle_len - 1).to(device) + plan.sel_lo  # :324-326
            new_plans[li] = _planner.LayerPlan(_planner.GATHER, plan.seq_len, sink=plan.sink, sel_lo=plan.sel_lo,
                                               sel_hi=plan.sel_hi, k_sel=count, tail=plan.tail,
                                               score=_planner.SCORE_GIVEN_INDEX if count > 0 else _planner.SCORE_NONE)
            if count > 0:
                given[li] = rows.to(torch.int32).view(1, 1, count).expand(batch, heads, count).contiguous()
        return new_plans, given, None


def update_manager(h2o_manager, attention_scores=None, attention_queries=None, skip_layers=()) -> None:
    """The manager update a compress call makes before it selects (reference :274-275): from attention probabilities,
    or — :class:`H2OScoreSlab` only — from a :class:`kvcompress.QueryCapture` of the forward that produced them."""
    if attention_queries is not None:
        if not isinstance(h2o_manager, H2OScoreSlab):
            raise ValueError("attention_queries needs an H2OScoreSlab manager: H2OAttentionManager takes attention "
                             "probabilities (attention_scores) only")
        if attention_scores is not None:
            raise ValueError("pass attention_scores or attention_queries, not both")
        cap = attention_queries
        h2o_manager.update_from_queries(cap.queries, cap.keys, cap.masks, cap.scaling, list(skip_layers))
    elif h2o_manager is not None and attention_scores is not None:
        h2o_manager.update_attention_scores(attention_scores, list(skip_layers))


def check_carry(h2o_manager, carry_scores: Optional[bool]) -> None:
    """``carry_scores`` of a compress call (None: the manager's own setting) must agree with the manager: cumulative
    scores need an ``H2OScoreSlab(carry_scores=True)``; the torch manager keeps the reference's reset semantics."""
    if carry_scores is None:
        return
    carries = isinstance(h2o_manager, H2OScoreSlab) and h2o_manager.carry_scores
    if bool(carry_scores) != carries:
        raise ValueError(f"carry_scores={carry_scores} needs an h2o_manager that "
                         f"{'is H2OScoreSlab(carry_scores=True)' if carry_scores else 'does not carry its scores'}; "
                         f"got {type(h2o_manager).__name__}"
                         + (f"(carry_scores={h2o_manager.carry_scores})" if isinstance(h2o_manager, H2OScoreSlab) else ""))


def h2o_attention_compress(past_key_values, attention_scores=None, h2o_manager: Optional[H2OAttentionManager] = None,
                           start_size: int = 4, heavy_hitter_size: int = 64, recent_size: int = 444,
                           skip_layers: List[int] = [], attention_queries=None, carry_scores: Optional[bool] = None,
                           **kwargs) -> List[Tuple[torch.Tensor, torch.Tensor]]:
    """Sinks + heavy hitters + recent window; heavy hitters come from ``h2o_manager`` when given,
    otherwise from the lowest key norms (identical to ``h2o_l2_compress``).  ``attention_queries``: a
    :class:`kvcompress.QueryCapture` to update an :class:`H2OScoreSlab` from, instead of ``attention_scores``.

    Reset semantics (the reference's): the caller resets the manager after the compression.  Cumulative semantics:
    with ``H2OScoreSlab(carry_scores=True)`` the manager's accumulators are compacted in place with the kept rows, in
    the gather launch itself, and the caller does not reset (update once per forward, then compress without passing the
    scores again).  ``carry_scores`` (default: the manager's setting) must agree with the manager."""
    check_carry(h2o_manager, carry_scores)
    layers = as_layer_list(past_key_values)
    if not layers:
        return layers
    if h2o_manager is None:
        if attention_queries is not None:
            raise ValueError("attention_queries needs an H2OScoreSlab manager (h2o_manager=)")
        return h2o_l2_compress(layers, start_size, heavy_hitter_size, recent_size, skip_layers)
    keys = layers[0][0]
    return compress_with_manager(partial(_engine.run_plans, layers), seq_lens(layers),
                                 (keys.size(0), keys.size(1), keys.dtype, keys.device), h2o_manager, start_size,
                                 heavy_hitter_size, recent_size, skip_layers, attention_scores, attention_queries)


def compress_with_manager(run, lens, shape, h2o_manager, start_size: int, heavy_hitter_size: int, recent_size: int,
                          skip_layers, attention_scores=None, attention_queries=None):
    """h2o_attention with a manager, for the function and ``KVSlabCache.compress_``: update the manager, plan ``lens``,
    let the manager rewrite the plans for a ``(batch, heads, dtype, device)`` cache, compact with ``run(plans,
    given_indices=, given_scores=, carry=)`` (``run_plans`` or ``apply_plans_``) and book what was carried."""
    update_manager(h2o_manager, attention_scores, attention_queries, skip_layers)
    plans = cached_plans(_planner.plan_h2o, lens, start_size, heavy_hitter_size, recent_size, skip_layers=skip_layers)
    plans, given, scores, *carry = h2o_manager.compress_plans(plans, start_size, heavy_hitter_size, recent_size, *shape)
    carry = carry[0] if carry else None
    out = run(plans, given_indices=given, given_scores=scores, carry=carry)
    if carry is not None:
        h2o_manager.carried(plans, carry)
    return out


class _AccumulatorViews(Mapping):
    """``accumulated_attention`` of an :class:`H2OScoreSlab`: layer -> ``[B, Hq, key_len]`` view of the device
    accumulators (read-only: the next update overwrites them in place)."""

    def __init__(self, owner: "H2OScoreSlab"):
        self._owner = owner

    def __getitem__(self, layer_idx: int) -> torch.Tensor:
        n = self._owner._lens[layer_idx]
        return self._owner._acc[layer_idx, :, :, :n]

    def __iter__(self):
        return iter(sorted(self._owner._lens))

    def __len__(self) -> int:
        return len(self._owner._lens)


class H2OScoreSlab:
    """Device-resident H2O score bookkeeping: a drop-in for :class:`H2OAttentionManager` (same constructor
    arguments plus ``capacity``, same methods) wherever ``h2o_manager=`` is accepted.

    The decayed accumulators live in one ``[num_layers, B, Hq, capacity]`` buffer next to one
    ``[num_layers, B, capacity]`` buffer of head-summed score rows, both in the attention dtype, allocated on the
    first update and doubled when a ``key_len`` exceeds ``capacity``.  ``update_attention_scores`` is ONE
    ``kvc_h2o_accumulate`` launch for every layer it updates: the accumulator update with the reference's rounding
    points (bit-identical to the torch manager for one query per step) and the score row of the heavy-hitter region
    ``[start_size, key_len - recent_size)``.  At compression the score row is handed to the compaction as
    ``KVC_SCORE_GIVEN_SCORE_SHARED``: each batch entry keeps its own heavy hitters, shared by its KV heads (the sum
    runs over all ``Hq`` query heads, so GQA models need nothing else).  The host decides everything from integers it
    holds — no ``.item()``, no synchronisation.  ``reset`` touches no device memory.

    ``carry_scores=False`` (reset semantics, the reference's): the accumulators describe rows by position, so the
    caller resets the manager after every compression.  ``carry_scores=True`` (cumulative semantics): every compaction
    through this manager also moves the accumulator rows of every compressed layer it holds data for with their tokens
    — ``acc[:, h*G+g, i] = acc[:, h*G+g, src(i)]`` in the same launch that moves K and V — after which the layer holds
    ``C`` valid entries and its next update decays them and zero-extends the new row.  The caller then never resets:
    keys are ranked by the decayed attention they have received over the whole generation.

    ``tensor_cores=True`` sends every :meth:`update_from_queries` through ``kvc_h2o_accumulate_qk_tc``: the logits come
    from the tensor cores (16-bit q and K, fp32 accumulation) and the exponentials from ``exp2``, so its bits differ from
    the default CUDA-core form (both stay within 2 ulps of fp64 logits).  It is the form to use for prompt-sized query
    counts; bf16 / f16 models with head_dim 64, 80 or 128 only (``ValueError`` otherwise)."""

    def __init__(self, start_size: int = 4, heavy_hitter_size: int = 64, recent_size: int = 444,
                 num_layers: int = 32, num_heads: int = 32, decay_factor: float = 0.9, device=None,
                 capacity: Optional[int] = None, carry_scores: bool = False, tensor_cores: bool = False):
        self.start_size = start_size
        self.heavy_hitter_size = heavy_hitter_size
        self.recent_size = recent_size
        self.total_cache_size = start_size + heavy_hitter_size + recent_size
        self.num_layers = num_layers
        self.num_heads = num_heads
        self.decay_factor = decay_factor
        self.device = device
        self.capacity = capacity
        self.carry_scores = bool(carry_scores)
        self.tensor_cores = bool(tensor_cores)
        self.current_seq_len = 0
        self._acc: Optional[torch.Tensor] = None    # [L, B, Hq, capacity]
        self._score: Optional[torch.Tensor] = None  # [L, B, capacity]; row l holds [B, hi - lo] densely
        self._lens: Dict[int, int] = {}             # layer -> valid accumulator entries (the torch manager's size(-1))
        self._scored: Dict[int, Tuple[int, int]] = {}  # layer -> (lo, hi) its score row currently holds
        self._gen = 0                               # bumped whenever the buffers are reallocated
        self._plan_cache: Dict[tuple, tuple] = {}
        self._ws: Optional[torch.Tensor] = None     # workspace of update_from_queries (uint8)
        self._reorder_recs: Optional[tuple] = None  # (_gen, RegionRecords) of the accumulators, built by a reorder

    @property
    def accumulated_attention(self) -> Mapping:
        return _AccumulatorViews(self)

    def reset(self) -> None:
        self._lens = {}
        self._scored = {}
        self.current_seq_len = 0

    # ------------------------------------------------------------------ buffers
    def _ensure(self, batch: int, heads: int, dtype: torch.dtype, device: torch.device, need: int) -> None:
        acc = self._acc
        if acc is not None and (acc.shape[1:3] != (batch, heads) or acc.dtype != dtype or acc.device != device):
            if self._lens:
                raise ValueError(f"H2OScoreSlab: attention [B={batch}, Hq={heads}] {dtype} on {device} does not match "
                                 f"the accumulators [B={acc.size(1)}, Hq={acc.size(2)}] {acc.dtype} on {acc.device}; "
                                 "call reset() first")
            acc = None
        if acc is None:
            cap = max(self.capacity or 0, need, 1)
        elif need > acc.size(3):
            cap = acc.size(3)
            while cap < need:
                cap *= 2
        else:
            return
        new_acc = torch.empty((self.num_layers, batch, heads, cap), dtype=dtype, device=device)
        if acc is not None:
            new_acc[..., :acc.size(3)].copy_(acc)
        # score rows are dense [B, region] inside a row of the buffer: they do not survive a change of pitch, and are
        # produced again by the update that follows or, for the other layers, at the next compression
        self._acc, self.capacity = new_acc, cap
        self._score = torch.empty((self.num_layers, batch, cap), dtype=dtype, device=device)
        self._scored = {}
        self._gen += 1
        self._plan_cache.clear()

    def _score_row(self, layer_idx: int, batch: int, region: int) -> torch.Tensor:
        return self._score[layer_idx].view(-1)[:batch * region].view(batch, region)

    def _rescore(self, layers: List[Tuple[int, int, int]]) -> None:
        """Score rows of [lo, hi) from the accumulators as they are (attn = NULL), every layer in one launch."""
        recs = []
        for li, lo, hi in layers:
            n = self._lens[li]
            recs.append((None, self._acc[li], self._score[li], n, n, lo, hi))
            self._scored[li] = (lo, hi)
        _engine.h2o_accumulate(recs, self.decay_factor)

    def _takes(self, layer_idx: int, skip_layers, missing: bool) -> bool:
        """Whether an update takes a layer (not skipped, no input missing); refuses one past ``num_layers``."""
        if missing or layer_idx in skip_layers:
            return False
        if layer_idx >= self.num_layers:
            raise ValueError(f"H2OScoreSlab: layer {layer_idx} >= num_layers={self.num_layers}")
        return True

    def _record(self, layers: List[Tuple[int, int]], like: torch.Tensor) -> List[tuple]:
        """Book an update of ``(layer_idx, key_len)`` pairs from ``[B, Hq, ...]`` tensors like ``like``; returns
        ``(acc, score_out, prev_len, lo, hi)`` per layer for the launch records."""
        self._ensure(like.size(0), like.size(1), like.dtype, like.device, max(n for _, n in layers))
        out = []
        for layer_idx, key_len in layers:
            lo, hi, _ = _planner.h2o_score_region(key_len, key_len, self.start_size, self.heavy_hitter_size,
                                                  self.recent_size)
            out.append((self._acc[layer_idx], self._score[layer_idx], self._lens.get(layer_idx, -1), lo, hi))
            self._lens[layer_idx] = key_len
            self._scored[layer_idx] = (lo, hi)
            self.current_seq_len = key_len
        return out

    # ------------------------------------------------------------------ the manager's interface
    def update_attention_scores(self, attentions, skip_layers: List[int] = []) -> None:
        """acc <- decay * acc (zero-extended, or reset if the cache shrank) + attn.sum(query dim), and the score row of
        [start_size, key_len - recent_size) — one launch for every non-skipped, non-``None`` layer."""
        if attentions is None:
            return
        work = []
        for layer_idx, attn in enumerate(attentions):
            if not self._takes(layer_idx, skip_layers, attn is None):
                continue
            if attn.dim() != 4:
                raise ValueError(f"layer {layer_idx}: attention must be [B, Hq, n_query, key_len]")
            work.append((layer_idx, attn if attn.stride(-1) == 1 else attn.contiguous()))
        if not work:
            return
        _engine._require_cuda(work[0][1], "attention")
        booked = self._record([(layer_idx, attn.size(3)) for layer_idx, attn in work], work[0][1])
        _engine.h2o_accumulate([(attn, acc, score, prev_len, attn.size(3), lo, hi)
                                for (_, attn), (acc, score, prev_len, lo, hi) in zip(work, booked)], self.decay_factor)

    def _workspace(self, nbytes: int, device: torch.device) -> torch.Tensor:
        """The query path's workspace: kept between updates, grown by doubling, so a steady step allocates nothing."""
        ws = self._ws
        if ws is None or ws.device != device or ws.numel() < nbytes:
            cap = max(ws.numel() if ws is not None and ws.device == device else 0, 4096)
            while cap < nbytes:
                cap *= 2
            ws = self._ws = torch.empty((cap,), dtype=torch.uint8, device=device)
        return ws

    def update_from_queries(self, queries, keys, masks=None, scaling=None, skip_layers: List[int] = []) -> None:
        """The update of :meth:`update_attention_scores` with the attention probabilities rebuilt on the device from the
        post-RoPE ``queries[l]`` ``[B, Hq, T, D]`` and the cached ``keys[l]`` ``[B, Hkv, key_len, D]`` (any view whose
        rows are dense, e.g. a slab view) — the model never has to return attention weights.  ``masks[l]``: ``None``
        (causal: the queries are the last T positions) or a bool ``[B, 1, T, key_len]`` / ``[B, T, key_len]`` mask,
        True = visible.  ``scaling``: the logit scale, one float or one per layer (default ``D ** -0.5``).  The
        probabilities are ``softmax(fp32 logits).to(dtype)``: HF eager attention in a 16-bit model rounds the logits to
        the model dtype first, SDPA and flash do not.  Two launches for every non-skipped layer with queries and keys
        (three with ``tensor_cores=True``: statistics, column sums, score rows);
        no synchronisation (:func:`kvcompress.capture_queries` records these arguments from a model's forward)."""
        if queries is None:
            return
        work = []
        for layer_idx, q in enumerate(queries):
            k = keys[layer_idx] if layer_idx < len(keys) else None
            if not self._takes(layer_idx, skip_layers, q is None or k is None):
                continue
            if q.dim() != 4 or k.dim() != 4 or k.size(1) == 0 or q.size(1) % k.size(1):
                raise ValueError(f"layer {layer_idx}: queries must be [B, Hq, T, D] and keys [B, Hkv, key_len, D] with "
                                 f"Hkv dividing Hq, got {tuple(q.shape)} and {tuple(k.shape)}")
            mask = None if masks is None or layer_idx >= len(masks) else masks[layer_idx]
            if mask is not None:
                if mask.dim() == 4:
                    if mask.size(1) != 1:
                        raise ValueError(f"layer {layer_idx}: a per-head mask {tuple(mask.shape)} is not supported; "
                                         "pass [B, 1, T, key_len] or [B, T, key_len]")
                    mask = mask[:, 0]
                if mask.dtype != torch.bool:
                    raise ValueError(f"layer {layer_idx}: the mask must be bool (True = visible), got {mask.dtype}")
                if mask.dim() == 3 and mask.size(0) == 1 and q.size(0) > 1:
                    mask = mask.expand(q.size(0), -1, -1)
                if mask.dim() == 3 and mask.size(2) > k.size(2):
                    mask = mask[:, :, :k.size(2)]
                if mask.dim() == 3 and mask.size(2) > 1 and mask.stride(2) != 1:
                    mask = mask.contiguous()
            s = scaling[layer_idx] if isinstance(scaling, (list, tuple)) else scaling
            work.append((layer_idx, q if q.stride(-1) == 1 else q.contiguous(), k, mask,
                         q.size(3) ** -0.5 if s is None else float(s)))
        if not work:
            return
        q0, k0 = work[0][1], work[0][2]
        _engine._require_cuda(q0, "queries")
        if self.tensor_cores:
            if q0.dtype not in (torch.bfloat16, torch.float16):
                raise ValueError(f"H2OScoreSlab(tensor_cores=True): {q0.dtype} queries; the tensor-core form takes "
                                 "bfloat16 / float16 (use tensor_cores=False for float32)")
            if q0.size(3) not in (64, 80, 128):
                raise ValueError(f"H2OScoreSlab(tensor_cores=True): head_dim {q0.size(3)} is not 64, 80 or 128 (use "
                                 "tensor_cores=False)")
        booked = self._record([(layer_idx, k.size(2)) for layer_idx, _, k, _, _ in work], q0)
        recs = [(q, k, mask, acc, score, prev_len, lo, hi, s)
                for (_, q, k, mask, s), (acc, score, prev_len, lo, hi) in zip(work, booked)]
        update = _engine.h2o_accumulate_qk_tc if self.tensor_cores else _engine.h2o_accumulate_qk
        update(recs, self.decay_factor, q0.size(1) // k0.size(1), lambda n: self._workspace(n, q0.device))

    def get_heavy_hitter_indices(self, layer_idx: int, seq_len: int) -> torch.Tensor:
        """Indices (relative to the middle region, ascending) of its heaviest tokens — what
        :meth:`H2OAttentionManager.get_heavy_hitter_indices` returns, selected on the device (``kvc_select``)."""
        n = self._lens.get(layer_idx)
        if n is None:
            rows = _evenly_spaced(seq_len, self.start_size, self.heavy_hitter_size, self.recent_size)
            return torch.arange(rows.start, rows.stop, rows.step)
        lo, hi, k = _planner.h2o_score_region(seq_len, n, self.start_size, self.heavy_hitter_size, self.recent_size)
        if k == 0:
            return torch.tensor([], dtype=torch.long, device=self._acc.device)
        if self._scored.get(layer_idx) != (lo, hi):
            self._rescore([(layer_idx, lo, hi)])
        batch = self._acc.size(1)
        top = _engine.select(self._score_row(layer_idx, batch, hi - lo), k, largest=True).long()
        return top.squeeze(0) if batch == 1 else top

    # ------------------------------------------------------------------ compaction
    def _check_cache(self, batch: int, heads: int, dtype: torch.dtype, device: torch.device) -> None:
        """The accumulators against the cache a compaction runs on: the same dtype, batch and device and, to carry them
        with the rows, ``heads`` dividing their ``Hq``."""
        acc = self._acc
        if acc.dtype != dtype:
            raise ValueError(f"H2OScoreSlab: the attention dtype {acc.dtype} differs from the cache dtype {dtype}")
        if acc.size(1) != batch or acc.device != device or (self.carry_scores and acc.size(2) % heads):
            raise ValueError(f"H2OScoreSlab: accumulators of batch {acc.size(1)} with Hq={acc.size(2)} on "
                             f"{acc.device}, cache of batch {batch} with Hkv={heads} on {device}")

    def compress_plans(self, plans, start_size: int, heavy_hitter_size: int, recent_size: int, batch: int, heads: int,
                       dtype: torch.dtype, device):
        """The h2o plans rewritten with this manager's heavy hitters (reference h2o_attention.py:318-331) for a cache
        of ``[batch, heads, S, D]`` ``dtype`` layers.  Returns ``(PlanSet, given_indices, given_scores)``: layers with
        accumulated scores rank ``[sel_lo, sel_lo + region)`` by their score row (``SCORE_GIVEN_SCORE_SHARED``), layers
        without data since the last reset keep evenly spaced rows (``SCORE_GIVEN_INDEX``), an empty region keeps no
        heavy hitter.  Score rows whose region differs from the last update's are re-scored in one launch.
        With ``carry_scores=True`` a fourth item follows: ``{layer: (acc, group, prev_len)}`` for every compressed layer
        this manager holds accumulators for (``run_plans`` / ``apply_plans_`` ``carry=``); after the launch, hand the
        plans and that dict to :meth:`carried`."""
        device = torch.device(device)
        carry = None
        if self.carry_scores:
            carry = {}
            held = [li for li in plans.gather if li in self._lens]
            if held:
                self._check_cache(batch, heads, dtype, device)
                self._ensure(batch, self._acc.size(2), dtype, device, max(plans.plans[li].seq_len for li in held))
                group = self._acc.size(2) // heads
                carry = {li: (self._acc[li], group, self._lens[li]) for li in held}
        checked = carry is not None  # every layer scored below is held, so checked above
        decisions, rescore = [], []
        for li in plans.gather:
            p = plans.plans[li]
            if p.region == 0:
                decisions.append(None)
                continue
            S, middle_len = p.seq_len, p.sel_hi - p.sel_lo
            n = self._lens.get(li)
            if n is None:
                picked = _evenly_spaced(S, self.start_size, self.heavy_hitter_size, self.recent_size)
                decisions.append(("even", picked[:min(heavy_hitter_size, middle_len)]))
                continue
            lo, hi, k = _planner.h2o_score_region(S, n, self.start_size, self.heavy_hitter_size, self.recent_size)
            if k == 0:
                decisions.append(("none",))
                continue
            region = hi - lo
            count = min(k, heavy_hitter_size, middle_len)  # :321
            if count != k or region > middle_len:
                raise ValueError(f"layer {li}: H2OScoreSlab(start_size={self.start_size}, heavy_hitter_size="
                                 f"{self.heavy_hitter_size}, recent_size={self.recent_size}) selects {k} of {region} rows, "
                                 f"the compression keeps {count} of {middle_len}: use the same sizes for both")
            if not checked:
                self._check_cache(batch, heads, dtype, device)
                checked = True
            if self._scored.get(li) != (lo, hi):
                rescore.append((li, lo, hi))
            decisions.append(("score", region, count))
        if rescore:
            self._rescore(rescore)
        key = (id(plans), self._gen, batch, heads, device, tuple(decisions))
        hit = self._plan_cache.get(key)
        if hit is not None and hit[0] is plans:
            return hit[1:] if carry is None else hit[1:] + (carry,)
        new_plans, given, scores = list(plans.plans), {}, {}
        for li, d in zip(plans.gather, decisions):
            if d is None:
                continue
            p = plans.plans[li]
            middle_len = p.sel_hi - p.sel_lo
            count, score, sel_hi = 0, _planner.SCORE_NONE, p.sel_hi
            if d[0] == "even" and d[1]:
                picked = d[1]
                count = len(picked)
                rows = [min(max(x, 0), middle_len - 1) + p.sel_lo for x in picked]
                if any(b <= a for a, b in zip(rows, rows[1:])):
                    raise ValueError(f"layer {li}: evenly spaced rows {rows[:4]}... collide after clamping into the "
                                     f"region of {middle_len} rows")
                given[li] = (torch.arange(picked.start, picked.stop, picked.step, device=device, dtype=torch.int32)
                             .clamp_(0, middle_len - 1).add_(p.sel_lo)
                             .view(1, 1, count).expand(batch, heads, count).contiguous())
                score = _planner.SCORE_GIVEN_INDEX
            elif d[0] == "score":
                _, region, count = d
                sel_hi = p.sel_lo + region
                scores[li] = self._score_row(li, batch, region)
                score = _planner.SCORE_GIVEN_SCORE_SHARED
            new_plans[li] = _planner.LayerPlan(_planner.GATHER, p.seq_len, sink=p.sink, sel_lo=p.sel_lo, sel_hi=sel_hi,
                                               k_sel=count, tail=p.tail, score=score)
        ps = _engine.PlanSet(new_plans)
        if len(self._plan_cache) > 64:
            self._plan_cache.clear()
        self._plan_cache[key] = (plans, ps, given or None, scores or None)
        if carry is not None:
            return ps, given or None, scores or None, carry
        return ps, given or None, scores or None

    def _reorder_records(self, batch: int, device: torch.device) -> bytes:
        """``kvc_batch_region`` records of the valid accumulator entries ``[0, _lens[l])`` of every layer, for a batch
        reorder (none before the first update).  Pointers and strides are packed once per accumulator buffer (``_gen``
        changes whenever it is reallocated); each call writes the entries from ``_lens``.  Score rows are not moved:
        they are marked stale and rebuilt from the moved accumulators by the next update or compression."""
        self._scored = {}
        acc = self._acc
        if acc is None or not self._lens:
            return b""
        if acc.size(1) != batch or acc.device != torch.device(device):
            raise ValueError(f"H2OScoreSlab: accumulators of batch {acc.size(1)} on {acc.device}, reordered with a cache "
                             f"of batch {batch} on {device}")
        e = acc.element_size()
        if self._reorder_recs is None or self._reorder_recs[0] != self._gen:
            self._reorder_recs = (self._gen, _engine.RegionRecords(
                [(acc[l].data_ptr(), acc.stride(1) * e, acc.stride(2) * e, 0, acc.size(2), e)
                 for l in range(self.num_layers)]))
        return self._reorder_recs[1].packed([self._lens.get(l, 0) * e for l in range(self.num_layers)])

    def reorder_(self, index) -> "H2OScoreSlab":
        """Beam search's reorder of the accumulators: batch entry b of every layer's valid entries becomes what entry
        ``index[b]`` held (``index_select(0, index)``), ONE ``kvc_batch_reorder`` launch — for the function path, where
        transformers reorders a ``DynamicCache`` and the scores must follow.  ``index`` as in
        :meth:`KVSlabCache.reorder_`, which takes this manager as a follower to move it in the slab's launch.  A
        manager with no accumulators yet moves nothing."""
        if self._acc is None or not self._lens:
            self._scored = {}
            return self
        batch, device = self._acc.size(1), self._acc.device
        recs = self._reorder_records(batch, device)
        _engine.batch_reorder(recs, _engine.reorder_index(index, batch, device), batch)
        return self

    def carried(self, plans, carry: dict) -> None:
        """Bookkeeping after a compaction that carried ``carry`` (from :meth:`compress_plans`) with ``plans``: each
        carried layer now holds ``C`` valid entries, and its score row is stale."""
        for li in carry:
            self._lens[li] = plans.plans[li].out_len
            self._scored.pop(li, None)


def create_h2o_manager_from_model(model, **kwargs) -> H2OAttentionManager:
    """Manager sized from ``model.config`` (reference h2o_attention.py:366-391)."""
    config = model.config
    return H2OAttentionManager(
        start_size=kwargs.get("start_size", 4),
        heavy_hitter_size=kwargs.get("heavy_hitter_size", 64),
        recent_size=kwargs.get("recent_size", 444),
        num_layers=getattr(config, "num_hidden_layers", 32),
        num_heads=getattr(config, "num_attention_heads", 32),
        decay_factor=kwargs.get("decay_factor", 0.9),
        device=next(model.parameters()).device,
    )


__all__ = ["H2OAttentionManager", "H2OScoreSlab", "h2o_attention_compress", "create_h2o_manager_from_model",
           "compress_with_manager", "update_manager", "check_carry"]
