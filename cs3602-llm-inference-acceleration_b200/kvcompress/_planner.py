"""Host planner: turns each compression method's arguments into per-layer keep-plans.

Every hot-path method of the reference reduces, per layer, to one descriptor

    keep rows [0, sink)  U  (k_sel rows of [sel_lo, sel_hi) ranked by a key)  U  [S - tail, S)

(SURVEY.md §8a).  The integers are computed here with plain Python ``int`` / ``float``
arithmetic, expression by expression as the reference computes them, so that output lengths
can never differ through a float-rounding or FMA difference.  Nothing in this module touches
a tensor: plans are built from sequence lengths alone and are unit-testable on CPU.

Reference line ranges are cited next to each rule.  Python slice semantics the reference
relies on implicitly (``x[:, :, -0:]`` is the whole tensor, ``x[:, :, :n]`` clips at S) are
reproduced with :func:`prefix_len` / :func:`suffix_len`.
"""

from __future__ import annotations

from dataclasses import dataclass
from math import ceil
from typing import List, Sequence

# score kinds — values match include/kvc.h (kvc_score_kind)
SCORE_NONE = 0
SCORE_L2_LOW = 1
SCORE_L2_HIGH = 2
SCORE_SNAPKV_POOL = 3
SCORE_GIVEN_INDEX = 4
SCORE_GIVEN_SCORE = 5
SCORE_GIVEN_SCORE_SHARED = 6  # GIVEN_SCORE with one [B, region] row per batch entry, shared by its heads

KEEP = "keep"      # layer is returned untouched (the same tensor objects)
VIEW = "view"      # layer is replaced by the view  x[:, :, -view_n:, :]  (no bytes move)
GATHER = "gather"  # layer goes through the CUDA gather-compaction


@dataclass(frozen=True)
class LayerPlan:
    kind: str
    seq_len: int = 0
    sink: int = 0
    sel_lo: int = 0
    sel_hi: int = 0
    k_sel: int = 0
    tail: int = 0
    score: int = SCORE_NONE
    pool_kernel: int = 1
    view_n: int = 0

    @property
    def out_len(self) -> int:
        if self.kind == KEEP:
            return self.seq_len
        if self.kind == VIEW:
            return suffix_len(self.seq_len, self.view_n)
        return self.sink + self.k_sel + self.tail

    @property
    def region(self) -> int:
        return self.sel_hi - self.sel_lo if self.k_sel > 0 else 0


def prefix_len(seq_len: int, n: int) -> int:
    """Number of rows in ``x[:, :, :n]`` for a tensor with ``seq_len`` rows."""
    return len(range(seq_len)[:n])


def suffix_len(seq_len: int, n: int) -> int:
    """Number of rows in ``x[:, :, -n:]`` (``-0:`` is the whole tensor)."""
    return len(range(seq_len)[-n:])


def _keep(seq_len: int) -> LayerPlan:
    return LayerPlan(KEEP, seq_len)


def _view(seq_len: int, n: int) -> LayerPlan:
    return LayerPlan(VIEW, seq_len, view_n=n)


def _nonneg(**named: int) -> None:
    for name, value in named.items():
        if value < 0:
            raise ValueError(f"{name} must be >= 0, got {value}")


def _sandwich(seq_len: int, start: int, lo: int, hi: int, k: int, recent: int, score: int,
              pool_kernel: int = 1) -> LayerPlan:
    """sinks x[:, :, :start] + k rows of [lo, hi) + recent window x[:, :, -recent:]."""
    return LayerPlan(GATHER, seq_len, sink=prefix_len(seq_len, start), sel_lo=lo, sel_hi=hi, k_sel=k,
                     tail=suffix_len(seq_len, recent) if recent is not None else 0, score=score if k > 0 else SCORE_NONE,
                     pool_kernel=pool_kernel)


# --------------------------------------------------------------------------- l2_compress
def plan_l2(seq_lens: Sequence[int], keep_ratio: float, prune_after: int, skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/l2_compress.py:48-65."""
    if keep_ratio >= 1.0:  # :48-49
        return [_keep(s) for s in seq_lens]
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if seq_len <= prune_after or layer_idx in skip_layers:  # :55-60
            plans.append(_keep(seq_len))
            continue
        tokens_to_keep = ceil(keep_ratio * seq_len)  # :62
        if tokens_to_keep >= seq_len:  # :64-65
            plans.append(_keep(seq_len))
            continue
        _nonneg(tokens_to_keep=tokens_to_keep)
        plans.append(LayerPlan(GATHER, seq_len, sel_lo=0, sel_hi=seq_len, k_sel=tokens_to_keep,
                               score=SCORE_L2_LOW if tokens_to_keep > 0 else SCORE_NONE))
    return plans


# --------------------------------------------------------------------------- fix_size_l2
_FIX_STRATEGIES = {"keep_low": SCORE_L2_LOW, "keep_high": SCORE_L2_HIGH, "random": SCORE_GIVEN_INDEX}


def plan_fix_size(seq_lens: Sequence[int], fix_kv_size: int, keep_ratio: float, strategy: str,
                  skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/fix_size_l2.py:65-147."""
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if seq_len <= fix_kv_size or layer_idx in skip_layers:  # :69-74
            plans.append(_keep(seq_len))
            continue
        protected = min(int(fix_kv_size * keep_ratio), seq_len)  # :79-80
        zone_end = seq_len - protected  # :83
        from_zone = fix_kv_size - protected  # :86
        if from_zone <= 0:  # :88-93 — protected recent rows only, as a view
            plans.append(_view(seq_len, protected))
            continue
        if zone_end <= from_zone:  # :95-97
            plans.append(_keep(seq_len))
            continue
        if strategy not in _FIX_STRATEGIES:  # :125-126
            raise ValueError(f"Unknown strategy: {strategy}")
        _nonneg(protected_length=protected)
        # :141-150 — the protected block is concatenated only when protected > 0
        plans.append(LayerPlan(GATHER, seq_len, sel_lo=0, sel_hi=zone_end, k_sel=from_zone, tail=protected,
                               score=_FIX_STRATEGIES[strategy]))
    return plans


# --------------------------------------------------------------------------- streaming_llm
def plan_streaming(seq_lens: Sequence[int], start_size: int, recent_size: int, skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/streaming_llm.py:83-109."""
    cache_size = start_size + recent_size
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if seq_len <= cache_size or layer_idx in skip_layers:  # :88-93
            plans.append(_keep(seq_len))
            continue
        _nonneg(start_size=start_size, recent_size=recent_size)
        plans.append(_sandwich(seq_len, start_size, 0, 0, 0, recent_size, SCORE_NONE))  # :99-107
    return plans


def plan_evict_for_space(seq_lens: Sequence[int], num_coming: int, start_size: int, recent_size: int,
                         skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/streaming_llm.py:143-168 (evict_for_space)."""
    cache_size = start_size + recent_size
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if seq_len + num_coming <= cache_size or layer_idx in skip_layers:  # :147-152
            plans.append(_keep(seq_len))
            continue
        effective_recent = recent_size - num_coming  # :155-157
        if effective_recent <= 0:
            effective_recent = recent_size
        _nonneg(start_size=start_size, effective_recent=effective_recent)
        plans.append(_sandwich(seq_len, start_size, 0, 0, 0, effective_recent, SCORE_NONE))
    return plans


# --------------------------------------------------------------------------- h2o_l2
def plan_h2o(seq_lens: Sequence[int], start_size: int, heavy_hitter_size: int, recent_size: int,
             skip_layers, score: int = SCORE_L2_LOW) -> List[LayerPlan]:
    """reference kvcompress/methods/h2o_l2.py:75-151."""
    total = start_size + heavy_hitter_size + recent_size
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if seq_len <= total or layer_idx in skip_layers:  # :81-86
            plans.append(_keep(seq_len))
            continue
        _nonneg(start_size=start_size, heavy_hitter_size=heavy_hitter_size, recent_size=recent_size)
        middle_start, middle_end = start_size, seq_len - recent_size  # :95-96
        if middle_end <= middle_start:  # :99-109 — sinks + recent only
            plans.append(_sandwich(seq_len, start_size, 0, 0, 0, recent_size, SCORE_NONE))
            continue
        num_to_keep = min(heavy_hitter_size, middle_end - middle_start)  # :125
        plans.append(_sandwich(seq_len, start_size, middle_start, middle_end, num_to_keep, recent_size, score))
    return plans


def h2o_score_region(seq_len: int, acc_len: int, start_size: int, heavy_hitter_size: int, recent_size: int):
    """reference h2o_attention.py:153-213 (get_heavy_hitter_indices): the heavy-hitter region ``[lo, hi)`` ranked by
    accumulators that cover ``acc_len`` keys when the cache holds ``seq_len`` rows, and the number of rows it yields.
    ``(0, 0, 0)`` when the region is empty."""
    lo, hi = start_size, min(seq_len, acc_len) - recent_size
    if hi <= lo:
        return 0, 0, 0
    return lo, hi, min(heavy_hitter_size, hi - lo)


# --------------------------------------------------------------------------- snapkv_lite
def plan_snapkv(seq_lens: Sequence[int], observation_window: int, keep_size: int, pooling_kernel: int,
                skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/snapkv_lite.py:66-152."""
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if seq_len <= keep_size or layer_idx in skip_layers:  # :70-75
            plans.append(_keep(seq_len))
            continue
        prefix = seq_len - observation_window  # :83
        if prefix <= 0:  # :84-86
            plans.append(_keep(seq_len))
            continue
        _nonneg(observation_window=observation_window)
        num_prefix = min(keep_size - observation_window, prefix)  # :125-126
        if num_prefix <= 0:  # :128-131 — observation window only, as a view
            plans.append(_view(seq_len, observation_window))
            continue
        plans.append(_sandwich(seq_len, 0, 0, prefix, num_prefix, observation_window, SCORE_SNAPKV_POOL,
                               pool_kernel=int(pooling_kernel)))
    return plans


# --------------------------------------------------------------------------- pyramid_kv
def pyramid_layer_sizes(num_layers: int, base_size: int, layer_decay: float, min_size: int, profile: str) -> List[int]:
    """Per-layer budgets, reference kvcompress/methods/pyramid_kv.py:84-97."""
    sizes = []
    for layer_idx in range(num_layers):
        if profile == "exponential":
            size = int(base_size * (layer_decay ** layer_idx))
        elif profile == "linear":
            decay_per_layer = (base_size - min_size) / max(num_layers - 1, 1)
            size = int(base_size - layer_idx * decay_per_layer)
        else:  # constant
            size = base_size
        sizes.append(max(size, min_size))
    return sizes


def _sinks_middle_recent(seq_len: int, target: int, start: int) -> LayerPlan:
    """Shared tail of pyramid_kv.py:115-181 and adaptive_l2.py:86-143."""
    recent = target // 2
    middle_to_keep = target - start - recent
    if middle_to_keep <= 0:  # pyramid :119-124 / adaptive :93-98 — last `target` rows, as a view
        return _view(seq_len, target)
    middle_start, middle_end = start, seq_len - recent
    if middle_end <= middle_start:  # pyramid :130-140 / adaptive :104-113
        return _sandwich(seq_len, start, 0, 0, 0, target - start, SCORE_NONE)
    num_to_keep = min(middle_to_keep, middle_end - middle_start)
    return _sandwich(seq_len, start, middle_start, middle_end, num_to_keep, recent, SCORE_L2_LOW)


def plan_pyramid(seq_lens: Sequence[int], base_size: int, layer_decay: float, min_size: int, profile: str,
                 skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/pyramid_kv.py:81-183."""
    sizes = pyramid_layer_sizes(len(seq_lens), base_size, layer_decay, min_size, profile)
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        target = sizes[layer_idx]
        if seq_len <= target or layer_idx in skip_layers:  # :104-109
            plans.append(_keep(seq_len))
            continue
        _nonneg(target_size=target)
        plans.append(_sinks_middle_recent(seq_len, target, min(4, target // 8)))  # :115
    return plans


# --------------------------------------------------------------------------- adaptive_l2
def plan_adaptive(seq_lens: Sequence[int], target_size: int, soft_limit: int, hard_limit: int, keep_ratio_min: float,
                  keep_ratio_max: float, skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/adaptive_l2.py:67-199."""
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if layer_idx in skip_layers or seq_len <= soft_limit:  # :71-77
            plans.append(_keep(seq_len))
            continue
        if seq_len > hard_limit:  # :81-145
            if seq_len <= target_size:
                plans.append(_keep(seq_len))
                continue
            _nonneg(target_size=target_size)
            plans.append(_sinks_middle_recent(seq_len, target_size, 4))
            continue
        # gradual zone :147-199
        progress = (seq_len - soft_limit) / (hard_limit - soft_limit)
        keep_ratio = keep_ratio_max - progress * (keep_ratio_max - keep_ratio_min)
        tokens_to_keep = max(int(seq_len * keep_ratio), soft_limit)
        if tokens_to_keep >= seq_len:
            plans.append(_keep(seq_len))
            continue
        protected_recent = int(tokens_to_keep * 0.2)
        from_history = tokens_to_keep - protected_recent
        if from_history <= 0:  # :163-168 — last tokens_to_keep rows, as a view
            plans.append(_view(seq_len, tokens_to_keep))
            continue
        selection_end = seq_len - protected_recent
        if selection_end <= from_history:  # :173-174
            plans.append(_keep(seq_len))
            continue
        _nonneg(protected_recent=protected_recent)
        plans.append(_sandwich(seq_len, 0, 0, selection_end, from_history, protected_recent, SCORE_L2_LOW))
    return plans


# --------------------------------------------------------------------------- recent_only
def plan_recent_only(seq_lens: Sequence[int], window_size: int, skip_layers) -> List[LayerPlan]:
    """reference kvcompress/methods/recent_only.py:53-68."""
    plans = []
    for layer_idx, seq_len in enumerate(seq_lens):
        if seq_len <= window_size or layer_idx in skip_layers:  # :57-62
            plans.append(_keep(seq_len))
            continue
        plans.append(_view(seq_len, window_size))  # :65-66
    return plans


def algorithmic_bytes(plans: Sequence[LayerPlan], batch: int, heads: int, head_dim: int, elem_bytes: int) -> int:
    """HBM bytes the path must move: e*B*H*D*(R + 4*C) per gathered layer (SURVEY.md §8d)."""
    rows = sum(p.region + 4 * p.out_len for p in plans if p.kind == GATHER)
    return rows * batch * heads * head_dim * elem_bytes
