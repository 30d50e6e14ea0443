"""KVSlabCache — the cache container for the decode loop: in-place append and in-place compression.

This is the step on both sides of the compress call (SURVEY.md §8f rank 1).  The reference's loop
(kvcompress/evaluate.py:132-166) re-allocates and copies the whole cache twice per generated token:

    outputs = model(token, past_key_values=cache)          # DynamicLayer.update: torch.cat per layer
    kv_list = list(normalize_kv_cache(outputs.past_key_values))
    compressed = compress_fn(kv_list, skip_layers=..., **kw)   # gather into fresh tensors (+ cat)
    cache = to_dynamic_cache(compressed)                    # reference utils.py:12-27

Here every layer's K and V live in pre-allocated ``[B, H, capacity, D]`` slabs on the GPU, next to a
``[B, H, capacity]`` array of key norms (what ``torch.norm(K, p=2, dim=-1)`` returns for those rows):

    cache.update(k_new, v_new, layer_idx)     # rows written in place, their norms recorded (one kernel)
    cache.compress_("h2o_l2", skip_layers=..., **kw)   # ONE launch for all layers, no allocation:
                                                       # scores from the stored norms, rows slide down

``compress_`` keeps exactly the rows the function of the same name keeps (same planner, same select,
bit-identical norms) — ``tests/test_gpu_slab.py`` walks both loops side by side.  Any registered
compress function also accepts a slab cache directly (``to_legacy_cache`` hands out views) and then ranks
rows from the stored norms (``key_norm_layers``) instead of re-reading K.

``pinned=True`` keeps the slabs — K, V **and the norms** — in page-locked HOST memory (an offloaded cache),
mapped into the GPU's address space: ``update`` writes new rows and their norms over PCIe, ``compress_`` and
the compress functions read 2-4 bytes per row for scoring and pull only the rows that are kept.
"""

from __future__ import annotations

import ctypes
import inspect
import struct
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _engine
from . import _planner as P

_SLAB = struct.Struct("3P6q")    # kvc_slab_layer: k v norms | k_stride_b k_stride_h v_stride_b v_stride_h n_stride_b n_stride_h
_ROWS = struct.Struct("2P6q2i")  # kvc_slab_new_rows: k_new v_new | 6 strides | cur_len n_new
assert _SLAB.size == 72 and _ROWS.size == 72

# method name -> (planner, planner arguments in order); defaults come from the compress function's signature
_PLANNERS = {
    "l2_compress": (P.plan_l2, ("keep_ratio", "prune_after")),
    "fix_size_l2": (P.plan_fix_size, ("fix_kv_size", "keep_ratio", "strategy")),
    "streaming_llm": (P.plan_streaming, ("start_size", "recent_size")),
    "recent_only": (P.plan_recent_only, ("window_size",)),
    "h2o_l2": (P.plan_h2o, ("start_size", "heavy_hitter_size", "recent_size")),
    "snapkv_lite": (P.plan_snapkv, ("observation_window", "keep_size", "pooling_kernel")),
    "pyramid_kv": (P.plan_pyramid, ("base_size", "layer_decay", "min_size", "profile")),
    "adaptive_l2": (P.plan_adaptive, ("target_size", "soft_limit", "hard_limit", "keep_ratio_min", "keep_ratio_max")),
}
_DEFAULTS: Dict[str, dict] = {}


def _method_defaults(method: str) -> dict:
    if method not in _DEFAULTS:
        from .methods import COMPRESS_METHODS

        sig = inspect.signature(COMPRESS_METHODS[method])
        _DEFAULTS[method] = {k: v.default for k, v in sig.parameters.items() if v.default is not inspect.Parameter.empty}
    return _DEFAULTS[method]


def _in_place(plans: Sequence[P.LayerPlan]) -> List[P.LayerPlan]:
    """A slab's valid rows always start at row 0, so a tail-only result (a view in the reference,
    e.g. recent_only.py:65-66) becomes a physical move of the last n rows."""
    out = []
    for p in plans:
        if p.kind == P.VIEW:
            out.append(P.LayerPlan(P.GATHER, p.seq_len, tail=P.suffix_len(p.seq_len, p.view_n)))
        else:
            out.append(p)
    return out


class KVSlabCache:
    """Pre-allocated per-layer K/V slabs with in-place ``update`` (append) and ``compress_``."""

    def __init__(self, num_layers: int, batch: int, heads: int, head_dim: int, capacity: int,
                 dtype: torch.dtype = torch.bfloat16, device="cuda", pinned: bool = False):
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("KVSlabCache runs on a CUDA device (sm_100a): there is no CPU path "
                               "(pinned=True keeps the slabs in host memory, the kernels still run on `device`)")
        if dtype not in _engine.KVC_DTYPE:
            raise ValueError(f"dtype {dtype} is not supported (float32, float16, bfloat16)")
        row_bytes = head_dim * torch.empty((), dtype=dtype).element_size()
        if row_bytes % 16 or not 16 <= row_bytes <= 2048:
            raise ValueError(f"head_dim*itemsize = {row_bytes} B: rows must be a multiple of 16 bytes, at most 2 KB")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        self.num_layers, self.batch, self.heads, self.head_dim = num_layers, batch, heads, head_dim
        self.capacity, self.dtype, self.device, self.pinned = capacity, dtype, device, bool(pinned)
        # `device` is where the kernels run; pinned slabs live in page-locked host memory mapped into its address space
        alloc = dict(dtype=dtype, pin_memory=True) if pinned else dict(dtype=dtype, device=device)
        # Pitch of one (batch, head) unit.  A pitch that is a multiple of 16 KB (4096 rows x 160 B = 640 KB, 32768 rows
        # x 256 B = 8 MB ...) puts the same rows of every unit on the same HBM channels: moving the 508-row tails of
        # 1024 such units runs at 0.91 of the copy peak with per-channel activity between 38 % and 83 %, and at 1.02
        # with 8 more rows of pitch (profiles/r02_stream_copy_control.json).  The reference's [B,H,S,D] tensors are
        # what they are; the slab owns its layout, so it pads.
        pitch = capacity
        while (pitch * row_bytes) % 16384 == 0:
            pitch += 8
        self.pitch = pitch
        self.k = torch.empty((num_layers, batch, heads, pitch, head_dim), **alloc)[:, :, :, :capacity]
        self.v = torch.empty((num_layers, batch, heads, pitch, head_dim), **alloc)[:, :, :, :capacity]
        self.n = torch.zeros((num_layers, batch, heads, capacity), **alloc)
        self.lengths: List[int] = [0] * num_layers
        self._shape = _engine._SHAPE.pack(batch, heads, head_dim, _engine.KVC_DTYPE[dtype], device.index)
        self._recs = [_SLAB.pack(self.k[l].data_ptr(), self.v[l].data_ptr(), self.n[l].data_ptr(),
                                 self.k.stride(1), self.k.stride(2), self.v.stride(1), self.v.stride(2),
                                 self.n.stride(1), self.n.stride(2)) for l in range(num_layers)]
        self._all_recs = b"".join(self._recs)
        self._k_layers = list(self.k.unbind(0))
        self._v_layers = list(self.v.unbind(0))
        self._lib = None
        self._fast_update = None   # compiled per-layer update (csrc/kvc_fast_binding.cpp), device slabs only
        if not pinned:
            mod = _engine.fast_binding()
            if mod is not None:
                lib = _engine.load_library()
                self._fast_update = mod.SlabFast(self._k_layers, self._v_layers, list(self.n.unbind(0)),
                                                 ctypes.cast(lib.kvc_slab_append, ctypes.c_void_p).value).update
        self._ws = None
        self._launch_cache: Dict[int, tuple] = {}

    # ------------------------------------------------------------------ construction / views
    @classmethod
    def from_legacy_cache(cls, past_key_values, capacity: Optional[int] = None, pinned: Optional[bool] = None,
                          device=None) -> "KVSlabCache":
        """Build a slab cache holding a list of ``(K, V)`` pairs (``capacity`` rows per layer, default: twice the
        longest layer).  ``pinned`` defaults to where the pairs live: host tensors give a pinned-host slab."""
        from .utils import normalize_kv_cache

        layers = list(normalize_kv_cache(past_key_values))
        if not layers:
            raise ValueError("cannot size a slab cache from an empty cache")
        k0 = layers[0][0]
        B, H, _, D = k0.shape
        longest = max(k.size(2) for k, _ in layers)
        if pinned is None:
            pinned = k0.device.type == "cpu"
        if device is None:
            device = k0.device if k0.is_cuda else torch.device("cuda", torch.cuda.current_device())
        cache = cls(len(layers), B, H, D, capacity or max(2 * longest, 16), k0.dtype, device, pinned=pinned)
        cache.append(layers)
        return cache

    def __len__(self) -> int:
        return self.num_layers

    def __getitem__(self, layer_idx: int) -> Tuple[torch.Tensor, torch.Tensor]:
        n = self.lengths[layer_idx]
        return self._k_layers[layer_idx].narrow(2, 0, n), self._v_layers[layer_idx].narrow(2, 0, n)

    def __iter__(self):
        return (self[l] for l in range(self.num_layers))

    def to_legacy_cache(self) -> List[Tuple[torch.Tensor, torch.Tensor]]:
        """Views of the valid rows, layer by layer — what ``normalize_kv_cache`` (reference utils.py:30-44) asks for."""
        return [self[l] for l in range(self.num_layers)]

    def get_seq_length(self, layer_idx: int = 0) -> int:
        return self.lengths[layer_idx] if self.num_layers else 0

    def key_norms(self, layer_idx: int) -> torch.Tensor:
        """Stored ``||K||_2`` of the valid rows of one layer, ``[B, H, S]`` in the cache dtype."""
        return self.n[layer_idx, :, :, :self.lengths[layer_idx]]

    def key_norm_layers(self) -> List[torch.Tensor]:
        """Per-layer stored norms for the compress functions (``methods/_common.stored_norms``)."""
        return [self.n[l, :, :, :self.lengths[l]] for l in range(self.num_layers)]

    def _finish(self) -> None:
        """Pinned slabs are read by the host with plain loads: finish the device work before returning, as the
        reference's (synchronous) CPU path does."""
        if self.pinned and not torch.cuda.is_current_stream_capturing():
            torch.cuda.current_stream(self.device).synchronize()

    def as_hf_cache(self):
        """This slab as a ``transformers.Cache``: the model's attention layers call ``update`` (in-place append)
        and read lengths / mask sizes from the slab, so it can be passed as ``past_key_values``."""
        from transformers.cache_utils import Cache, CacheLayerMixin

        slab = self

        class _SlabLayer(CacheLayerMixin):
            is_sliding = False
            is_compileable = False

            def __init__(self, layer_idx: int):
                self.layer_idx = layer_idx
                self.is_initialized = True
                self.dtype, self.device = slab.dtype, slab.device

            keys = property(lambda self: slab[self.layer_idx][0], lambda self, value: None)
            values = property(lambda self: slab[self.layer_idx][1], lambda self, value: None)

            def lazy_initialization(self, key_states, value_states) -> None:
                return None

            def update(self, key_states, value_states, *args, **kwargs):
                return slab.update(key_states, value_states, self.layer_idx)

            def get_mask_sizes(self, query_length) -> Tuple[int, int]:
                q = query_length if isinstance(query_length, int) else int(query_length.shape[0])
                return slab.lengths[self.layer_idx] + q, 0

            def get_seq_length(self) -> int:
                return slab.lengths[self.layer_idx]

            def get_max_cache_shape(self) -> int:
                return -1

            def reset(self) -> None:
                slab.lengths[self.layer_idx] = 0

        cache = Cache(layers=[_SlabLayer(l) for l in range(self.num_layers)])
        cache.slab = self
        return cache

    # ------------------------------------------------------------------ append
    def _check_new(self, keys: torch.Tensor, values: torch.Tensor, layer_idx: int) -> None:
        for t in (keys, values):
            if not (t.device == self.device or (t.device.type == "cpu" and t.is_pinned())):
                raise RuntimeError(f"layer {layer_idx}: new rows must live on {self.device} or in pinned host memory "
                                   f"(got {t.device}); there is no CPU path")
        if keys.dtype != self.dtype or values.dtype != self.dtype:
            raise ValueError(f"layer {layer_idx}: new rows must be {self.dtype}")
        if keys.dim() != 4 or keys.shape != values.shape or keys.size(0) != self.batch or keys.size(1) != self.heads \
                or keys.size(3) != self.head_dim:
            raise ValueError(f"layer {layer_idx}: new rows must be [B={self.batch}, H={self.heads}, T, D={self.head_dim}]")
        if self.lengths[layer_idx] + keys.size(2) > self.capacity:
            raise ValueError(f"layer {layer_idx}: {self.lengths[layer_idx]} + {keys.size(2)} rows exceed the slab "
                             f"capacity {self.capacity}")

    def _append(self, items: Sequence[Tuple[int, torch.Tensor, torch.Tensor]]) -> None:
        lib = _engine.load_library()
        slab_buf = bytearray(_SLAB.size * len(items))
        rows_buf = bytearray(_ROWS.size * len(items))
        keep = []
        host_temps = False  # pinned temporaries are not stream-ordered: the launch must finish before they are freed
        dt, dev, want = self.dtype, self.device, None
        for m, (l, keys, values) in enumerate(items):
            shape = keys.shape
            if want is None:
                want = (self.batch, self.heads, shape[2], self.head_dim) if len(shape) == 4 else None
            # one cheap comparison per tensor on the decode path; the detailed diagnosis only when it fails
            if not (keys.is_cuda and keys.dtype is dt and values.dtype is dt and keys.device == dev
                    and values.device == dev and tuple(shape) == want and values.shape == shape
                    and self.lengths[l] + shape[2] <= self.capacity):
                self._check_new(keys, values, l)
                want = None
            if not _engine._rows_ok(keys):
                host_temps = host_temps or not keys.is_cuda
                keys = keys.contiguous() if keys.is_cuda else keys.contiguous().pin_memory()
            if not _engine._rows_ok(values):
                host_temps = host_temps or not values.is_cuda
                values = values.contiguous() if values.is_cuda else values.contiguous().pin_memory()
            keep.append((keys, values))
            ks, vs = keys.stride(), values.stride()
            slab_buf[m * _SLAB.size:(m + 1) * _SLAB.size] = self._recs[l]
            _ROWS.pack_into(rows_buf, m * _ROWS.size, keys.data_ptr(), values.data_ptr(), ks[0], ks[1], ks[2],
                            vs[0], vs[1], vs[2], self.lengths[l], keys.size(2))
        status = lib.kvc_slab_append(self._shape, len(items), bytes(slab_buf), bytes(rows_buf),
                                     ctypes.c_void_p(_engine._stream_ptr(self.device)))
        _engine._check(status, "kvc_slab_append")
        for l, keys, _ in items:
            self.lengths[l] += keys.size(2)
        if host_temps and not self.pinned:
            torch.cuda.current_stream(self.device).synchronize()
        self._finish()

    def update(self, key_states: torch.Tensor, value_states: torch.Tensor, layer_idx: int, cache_kwargs=None):
        """HF ``Cache.update`` contract: append ``[B, H, T, D]`` rows to one layer, return that layer's full
        ``(K, V)`` (views of the slab) — replaces the ``torch.cat`` of transformers ``cache_utils.py:119-120``."""
        # hot path of the decode loop (called once per layer per token): the compiled binding validates, launches and
        # returns the views; None means "a case for the checks below" (wrong shape, capacity, host rows, ...)
        if self._fast_update is not None:
            n = self.lengths[layer_idx]
            done = self._fast_update(key_states, value_states, layer_idx, n)
            if done is not None:
                self.lengths[layer_idx] = n + key_states.shape[2]
                return done
        if not (key_states.is_cuda and key_states.dtype is self.dtype and value_states.dtype is self.dtype
                and key_states.device == self.device and value_states.device == self.device):
            self._check_new(key_states, value_states, layer_idx)
        shape = key_states.shape
        n, T = self.lengths[layer_idx], shape[2]
        if len(shape) != 4 or value_states.shape != shape or shape[0] != self.batch or shape[1] != self.heads \
                or shape[3] != self.head_dim or n + T > self.capacity:
            self._check_new(key_states, value_states, layer_idx)
        if T == 0:
            return self[layer_idx]
        host_temps = False
        if not _engine._rows_ok(key_states):
            host_temps = host_temps or not key_states.is_cuda
            key_states = key_states.contiguous() if key_states.is_cuda else key_states.contiguous().pin_memory()
        if not _engine._rows_ok(value_states):
            host_temps = host_temps or not value_states.is_cuda
            value_states = value_states.contiguous() if value_states.is_cuda else value_states.contiguous().pin_memory()
        ks, vs = key_states.stride(), value_states.stride()
        rows = _ROWS.pack(key_states.data_ptr(), value_states.data_ptr(), ks[0], ks[1], ks[2], vs[0], vs[1], vs[2], n, T)
        if self._lib is None:
            self._lib = _engine.load_library().kvc_slab_append
        status = self._lib(self._shape, 1, self._recs[layer_idx], rows, torch.cuda.current_stream(self.device).cuda_stream)
        if status:
            _engine._check(status, "kvc_slab_append")
        self.lengths[layer_idx] = n + T
        if host_temps and not self.pinned:
            torch.cuda.current_stream(self.device).synchronize()
        if self.pinned:
            self._finish()
        return self._k_layers[layer_idx].narrow(2, 0, n + T), self._v_layers[layer_idx].narrow(2, 0, n + T)

    def append(self, new_rows) -> "KVSlabCache":
        """Append one ``(k_new, v_new)`` pair per layer — every layer in ONE launch."""
        items = [(l, kv[0], kv[1]) for l, kv in enumerate(new_rows) if kv is not None and kv[0].size(2) > 0]
        if items:
            self._append(items)
        return self

    def append_stacked(self, k_new: torch.Tensor, v_new: torch.Tensor) -> "KVSlabCache":
        """Append ``[L, B, H, T, D]`` rows (one tensor for all layers, e.g. a model's fused KV projection output)
        in ONE launch; the per-layer host work is pointer arithmetic only."""
        if k_new.dim() != 5 or k_new.shape != v_new.shape or k_new.size(0) != self.num_layers:
            raise ValueError(f"stacked rows must be [L={self.num_layers}, B, H, T, D]")
        self._check_new(k_new[0], v_new[0], 0)
        T = k_new.size(3)
        if max(self.lengths) + T > self.capacity:
            raise ValueError(f"{max(self.lengths)} + {T} rows exceed the slab capacity {self.capacity}")
        host_temps = False
        if not (_engine._rows_ok(k_new[0]) and _engine._rows_ok(v_new[0])):
            host_temps = not k_new.is_cuda
            k_new, v_new = k_new.contiguous(), v_new.contiguous()
            if host_temps:  # .contiguous() of a pinned tensor is pageable: the GPU cannot read it
                k_new, v_new = k_new.pin_memory(), v_new.pin_memory()
        ks, vs, esz = k_new.stride(), v_new.stride(), k_new.element_size()
        kp, vp = k_new.data_ptr(), v_new.data_ptr()
        rows_buf = bytearray(_ROWS.size * self.num_layers)
        for l in range(self.num_layers):
            _ROWS.pack_into(rows_buf, l * _ROWS.size, kp + l * ks[0] * esz, vp + l * vs[0] * esz, ks[1], ks[2], ks[3],
                            vs[1], vs[2], vs[3], self.lengths[l], T)
        status = _engine.load_library().kvc_slab_append(self._shape, self.num_layers, self._all_recs, bytes(rows_buf),
                                                        ctypes.c_void_p(_engine._stream_ptr(self.device)))
        _engine._check(status, "kvc_slab_append")
        self.lengths = [n + T for n in self.lengths]
        if host_temps and not self.pinned:
            torch.cuda.current_stream(self.device).synchronize()
        self._finish()
        return self

    # ------------------------------------------------------------------ in-place compression
    def plans_for(self, method: str, **kwargs) -> _engine.PlanSet:
        """The in-place plans of ``COMPRESS_METHODS[method](cache, **kwargs)`` for the current lengths."""
        from .methods._common import cached_plans

        if method not in _PLANNERS:
            from .methods import COMPRESS_METHODS

            raise ValueError(f"Unknown method: {method}. Available in place: {list(_PLANNERS)}"
                             if method not in COMPRESS_METHODS else
                             f"{method} has no in-place form; call the function on the slab cache instead")
        planner, names = _PLANNERS[method]
        args = dict(_method_defaults(method))
        args.update(kwargs)
        return cached_plans(planner, self.lengths, *[args[n] for n in names], skip_layers=args.get("skip_layers", ()))

    def compress_(self, method: str, return_indices: bool = False, **kwargs):
        """``cache = to_dynamic_cache(get_compress_fn(method)(normalize_kv_cache(cache), **kwargs))`` in place:
        one launch for every layer, no allocation, scores from the stored key norms."""
        if method == "h2o_attention":
            return self._compress_h2o_attention(return_indices=return_indices, **kwargs)
        if method == "snapkv_lite" and kwargs.get("obs_queries") is not None:
            return self._compress_snapkv_vote(return_indices=return_indices, **kwargs)
        plans = self.plans_for(method, **kwargs)
        given = None
        if method == "fix_size_l2" and kwargs.get("strategy") == "random":
            from .methods.fix_size_l2 import _random_indices

            given = {li: _random_indices(self[li][0], p.sel_hi, p.k_sel)
                     for li, p in enumerate(plans) if p.kind == P.GATHER and p.score == P.SCORE_GIVEN_INDEX}
        return self.apply_plans_(plans, given_indices=given, return_indices=return_indices)

    def _compress_snapkv_vote(self, obs_queries, obs_lse=None, return_indices: bool = False, **kwargs):
        """snapkv_lite in vote mode, in place: the tcgen05 q.K^T vote over the slab's keys (one launch), then pool ->
        top-k -> slide inside the slab with the votes as caller-supplied scores (one launch).  Keeps the rows
        ``snapkv_lite_compress(cache, obs_queries=...)`` keeps."""
        from dataclasses import replace

        if self.pinned:
            raise RuntimeError("the q.K^T vote reads the keys through TMA tensor maps: device-resident slabs only")
        plans = self.plans_for("snapkv_lite", **kwargs)
        if len(obs_queries) != self.num_layers:
            raise ValueError(f"obs_queries: {len(obs_queries)} entries for {self.num_layers} layers")
        window = kwargs.get("observation_window", _method_defaults("snapkv_lite")["observation_window"])
        voted = [li for li, p in enumerate(plans) if p.kind == P.GATHER and p.k_sel > 0]
        for li in voted:
            if obs_queries[li] is None:
                raise ValueError(f"obs_queries[{li}] is missing for a layer that is compressed")
        scores = {}
        if voted:
            votes = _engine.snapkv_votes([(self[li][0], obs_queries[li]) for li in voted], window,
                                         lse=None if obs_lse is None else [obs_lse[li] for li in voted])
            scores = dict(zip(voted, votes))
        new_plans = [replace(p, score=P.SCORE_GIVEN_SCORE) if li in scores else p for li, p in enumerate(plans)]
        return self.apply_plans_(new_plans, given_scores=scores, return_indices=return_indices)

    def _compress_h2o_attention(self, attention_scores=None, h2o_manager=None, start_size: int = 4,
                                heavy_hitter_size: int = 64, recent_size: int = 444, skip_layers: Sequence[int] = (),
                                return_indices: bool = False, attention_queries=None,
                                carry_scores: Optional[bool] = None, **_ignored):
        """``h2o_attention_compress`` in place (reference h2o_attention.py:216-363): without a manager it is exactly
        ``h2o_l2`` (:337-351); with one, its head-summed heavy hitters are the caller-supplied rows of the in-place
        compaction (they must ascend strictly — the manager sorts them, a clamp collision is refused).
        ``attention_queries``: a ``QueryCapture`` that updates an ``H2OScoreSlab`` instead of ``attention_scores``.
        With ``H2OScoreSlab(carry_scores=True)`` the accumulators slide with the rows in the same launch (cumulative
        H2O); ``carry_scores`` (default: the manager's setting) must agree with the manager."""
        from .methods._common import cached_plans
        from .methods.h2o_attention import H2OScoreSlab, check_carry, manager_plans, update_manager

        check_carry(h2o_manager, carry_scores)
        if h2o_manager is None:
            if attention_queries is not None:
                raise ValueError("attention_queries needs an H2OScoreSlab manager (h2o_manager=)")
            return self.compress_("h2o_l2", return_indices=return_indices, start_size=start_size,
                                  heavy_hitter_size=heavy_hitter_size, recent_size=recent_size, skip_layers=skip_layers)
        update_manager(h2o_manager, attention_scores, attention_queries, skip_layers)
        plans = cached_plans(P.plan_h2o, self.lengths, start_size, heavy_hitter_size, recent_size, skip_layers=skip_layers)
        if isinstance(h2o_manager, H2OScoreSlab):  # scores ranked on the device: no host round trip
            plans, given, scores, *carry = h2o_manager.compress_plans(plans, start_size, heavy_hitter_size,
                                                                      recent_size, self.batch, self.heads, self.dtype,
                                                                      self.device)
            carry = carry[0] if carry else None
            res = self.apply_plans_(plans, given_indices=given, given_scores=scores, return_indices=return_indices,
                                    carry=carry)
            if carry is not None:
                h2o_manager.carried(plans, carry)
            return res
        plans, given = manager_plans(self.to_legacy_cache(), plans, h2o_manager, heavy_hitter_size)
        for li, rows in given.items():
            if rows.size(-1) > 1 and not bool((rows[0, 0, 1:] > rows[0, 0, :-1]).all()):
                raise ValueError(f"layer {li}: the manager's rows must ascend strictly for the in-place compaction")
        return self.apply_plans_(plans, given_indices=given, return_indices=return_indices)

    def evict_for_space_(self, num_coming: int, start_size: int = 4, recent_size: int = 508,
                         skip_layers: Sequence[int] = (), return_indices: bool = False):
        """``evict_for_space`` (reference streaming_llm.py:114-170) in place: make room for ``num_coming`` rows before
        a prefill chunk is appended — sinks stay where they are, the shortened recent window slides down behind them."""
        from .methods._common import cached_plans

        plans = cached_plans(P.plan_evict_for_space, self.lengths, num_coming, start_size, recent_size,
                             skip_layers=skip_layers)
        return self.apply_plans_(plans, return_indices=return_indices)

    def apply_plans_(self, plans, given_indices: Optional[dict] = None, return_indices: bool = False,
                     given_scores: Optional[dict] = None, carry: Optional[dict] = None):
        """Compact every GATHER layer of ``plans`` in place, in one launch.  ``carry``: {layer: (acc, group,
        prev_len)} per-row state that slides with the kept rows in the same launch (see :func:`_engine.run_plans`)."""
        ps = plans if isinstance(plans, _engine.PlanSet) else _engine.PlanSet(plans)
        if len(ps) != self.num_layers:
            raise ValueError(f"{len(ps)} plans for {self.num_layers} layers")
        entry = self._launch_cache.get(id(ps))
        if entry is None or entry[0] is not ps:
            moved = _in_place(ps.plans)
            ids = [i for i, p in enumerate(moved) if p.kind == P.GATHER]
            for i in ids:
                if moved[i].seq_len != self.lengths[i]:
                    raise ValueError(f"layer {i}: plan built for {moved[i].seq_len} rows, the slab holds {self.lengths[i]}")
            plan_buf = b"".join(_engine._PLAN.pack(p.seq_len, p.sink, p.sel_lo, p.sel_hi, p.k_sel, p.tail, p.score,
                                                   p.pool_kernel) for p in (moved[i] for i in ids))
            slab_buf = b"".join(self._recs[i] for i in ids)
            ws_need = int(_engine.load_library().kvc_workspace_bytes(self._shape, len(ids), plan_buf)) if ids else 0
            entry = (ps, ids, plan_buf, slab_buf, [moved[i].out_len for i in ids],
                     [moved[i].seq_len for i in ids], ws_need)
            if len(self._launch_cache) > 64:
                self._launch_cache.clear()
            self._launch_cache[id(ps)] = entry
        _, ids, plan_buf, slab_buf, out_lens, in_lens, ws_need = entry
        indices = {}
        if not ids:
            return (self, indices) if return_indices else self
        for i, n in zip(ids, in_lens):
            if self.lengths[i] != n:
                raise ValueError(f"layer {i}: plan built for {n} rows, the slab holds {self.lengths[i]}")
        idx_out = idx_in = None
        keep = []
        if return_indices:
            ptrs = (ctypes.c_void_p * len(ids))()
            for m, (i, c) in enumerate(zip(ids, out_lens)):
                t = torch.empty((self.batch, self.heads, c), dtype=torch.int32, device=self.device)
                indices[i] = t
                ptrs[m] = t.data_ptr()
            idx_out = ptrs
        if given_indices or given_scores:
            ptrs = (ctypes.c_void_p * len(ids))()
            for m, i in enumerate(ids):
                gs = given_scores.get(i) if given_scores else None
                if gs is not None:  # SCORE_GIVEN_SCORE(_SHARED): the region's scores travel in the idx_in slot (kvc.h)
                    want = _engine._score_shape(ps.plans[i], self.batch, self.heads)
                    if gs.dtype != self.dtype or not gs.is_contiguous() or gs.device != self.device \
                            or tuple(gs.shape) != want:
                        raise ValueError(f"layer {i}: scores must be a contiguous {self.dtype} {list(want)} tensor "
                                         f"on {self.device}")
                    keep.append(gs)
                    ptrs[m] = gs.data_ptr()
                    continue
                gi = given_indices.get(i) if given_indices else None
                if gi is not None:
                    if gi.device.type == "cpu" and self.pinned:
                        gi = gi.contiguous().pin_memory()  # drawn on the host for a host-resident slab
                    if gi.dtype != torch.int32 or not gi.is_contiguous() or (gi.device != self.device and not gi.is_pinned()):
                        raise ValueError(f"layer {i}: indices must be a contiguous int32 tensor on {self.device}")
                    keep.append(gi)
                    ptrs[m] = gi.data_ptr()
            idx_in = ptrs
        lib = _engine.load_library()
        ws_ptr = None
        if ws_need > 0:  # selection larger than shared memory (see kvc_workspace_bytes)
            if self._ws is None or self._ws.numel() < ws_need:
                self._ws = torch.empty((ws_need,), dtype=torch.uint8, device=self.device)
            ws_ptr = ctypes.c_void_p(self._ws.data_ptr())
        carry_buf = None  # a NULL carry is exactly kvc_slab_compress (kvc.h)
        if carry:
            carry_buf = b"".join(_engine.carry_record(i, carry[i], self.batch, self.heads, self.dtype, n)
                                 if carry.get(i) is not None else bytes(_engine._CARRY.size)
                                 for i, n in zip(ids, in_lens))
        status = lib.kvc_slab_compress_carry(self._shape, len(ids), plan_buf, slab_buf, idx_out, idx_in, carry_buf,
                                             ws_ptr, ws_need, ctypes.c_void_p(_engine._stream_ptr(self.device)))
        _engine._check(status, "kvc_slab_compress")
        for i, c in zip(ids, out_lens):
            self.lengths[i] = c
        self._finish()
        return (self, indices) if return_indices else self


class SlabDecodeStep:
    """One steady-state decode step — append one token per layer, compress in place — captured in a CUDA graph.

    At steady state every step has the same shape (``S = cap`` rows, one new row, ``cap`` rows kept), the slab's
    pointers never change and nothing is allocated, so the two launches replay from a graph with no per-step host
    work.  Write the new token's rows into ``k_new`` / ``v_new`` (``[L, B, H, 1, D]``, static buffers) and call the
    object; the slab is updated in place.  Built by :meth:`KVSlabCache.capture_step`."""

    def __init__(self, slab: "KVSlabCache", method: str, kwargs: dict):
        self.slab, self.method, self.kwargs = slab, method, dict(kwargs)
        L, B, H, D = slab.num_layers, slab.batch, slab.heads, slab.head_dim
        self.k_new = torch.zeros((L, B, H, 1, D), dtype=slab.dtype, device=slab.device)
        self.v_new = torch.zeros((L, B, H, 1, D), dtype=slab.dtype, device=slab.device)
        before = list(slab.lengths)
        if len(set(before)) != 1:
            raise ValueError("capture_step needs every layer at the same length (no skipped, growing layers)")
        saved = (slab.k.clone(), slab.v.clone(), slab.n.clone())
        stream = torch.cuda.Stream(device=slab.device)
        stream.wait_stream(torch.cuda.current_stream(slab.device))
        with torch.cuda.stream(stream):  # warm-up outside capture: library attributes, plan caches
            slab.append_stacked(self.k_new, self.v_new)
            slab.compress_(method, **self.kwargs)
        torch.cuda.current_stream(slab.device).wait_stream(stream)
        if slab.lengths != before:
            raise ValueError(f"{method}: a step changes the cache lengths {before} -> {slab.lengths}; capture at steady "
                             "state (the cache already at its cap)")
        slab.k.copy_(saved[0]), slab.v.copy_(saved[1]), slab.n.copy_(saved[2])
        del saved
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            slab.append_stacked(self.k_new, self.v_new)
            slab.compress_(method, **self.kwargs)
        # capture records, it does not run: lengths were advanced on the host only — they are the steady state
        assert slab.lengths == before

    def __call__(self) -> "KVSlabCache":
        self.graph.replay()
        return self.slab


def _capture_step(self, method: str, **kwargs) -> SlabDecodeStep:
    """Capture ``append_stacked(k_new, v_new); compress_(method, **kwargs)`` at steady state in a CUDA graph."""
    return SlabDecodeStep(self, method, kwargs)


KVSlabCache.capture_step = _capture_step

__all__ = ["KVSlabCache", "SlabDecodeStep"]
