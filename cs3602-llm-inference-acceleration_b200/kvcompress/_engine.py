"""ctypes binding to ``libkvc_sm100a.so`` (C ABI in ``include/kvc.h``) and plan execution.

This is the only module that talks to the device library.  There is no CPU path and no
fallback: if a plan needs data movement, the tensors must be reachable by the GPU — CUDA
tensors, or page-locked (pinned) host tensors, which the kernels read and write in place over
PCIe (an offloaded cache: only the rows a method needs ever cross the link) — and the shared
library must be present, otherwise a ``RuntimeError`` is raised.

PyTorch is used for device memory (``torch.empty`` through the caching allocator) and for
the current stream; all compute happens in the library's own sm_100a kernels.
"""

from __future__ import annotations

import ctypes
import os
import struct
from typing import List, Optional, Sequence, Tuple

import torch

from . import _planner as P

_LIB_NAME = "libkvc_sm100a.so"
_CSRC_DIR = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "csrc"))
_LIB_PATH = os.path.join(_CSRC_DIR, _LIB_NAME)

# struct layouts of include/kvc.h
_PLAN = struct.Struct("8i")        # kvc_layer_plan: seq_len sink sel_lo sel_hi k_sel tail score pool_kernel
_IO = struct.Struct("4P6q4P2q")    # kvc_layer_io: k_in v_in k_out v_out | 6 strides | idx_out idx_in score_in norms_in | 2 strides
_SHAPE = struct.Struct("5i")       # kvc_shape: batch heads head_dim dtype device
assert _PLAN.size == 32 and _IO.size == 128 and _SHAPE.size == 20
KVC_ABI_VERSION = 5

KVC_DTYPE = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}
KVC_OK = 0
_STATUS_EXC = {1: ValueError, 2: ValueError, 3: ValueError, 4: RuntimeError}

_RANKED = (P.SCORE_L2_LOW, P.SCORE_L2_HIGH, P.SCORE_SNAPKV_POOL)  # scores derived from key norms
_GIVEN_SCORES = (P.SCORE_GIVEN_SCORE, P.SCORE_GIVEN_SCORE_SHARED)  # scores supplied by the caller


_CARRY = struct.Struct("P2q2i")   # kvc_carry_layer: acc | acc_stride_b acc_stride_h | group prev_len
assert _CARRY.size == 32


def carry_record(li: int, spec, B: int, H: int, dtype, seq_len: int) -> bytes:
    """The ``kvc_carry_layer`` of layer ``li`` from ``(acc, group, prev_len)``: acc a ``[B, H * group, >= seq_len]``
    CUDA tensor of the cache dtype with a dense last dimension, compacted in place with the layer's kept rows."""
    acc, group, prev_len = spec
    group, prev_len = int(group), int(prev_len)
    if group < 1 or prev_len < 0:
        raise ValueError(f"layer {li}: carry group must be >= 1 and prev_len >= 0, got {group} and {prev_len}")
    if not acc.is_cuda or acc.dtype != dtype or acc.dim() != 3 or acc.size(0) != B or acc.size(1) != H * group \
            or acc.size(2) < seq_len or (acc.stride(2) != 1 and acc.size(2) > 1):
        raise ValueError(f"layer {li}: carried state must be a CUDA {dtype} [B={B}, H*group={H * group}, >= {seq_len}] "
                         "tensor with a dense last dimension")
    return _CARRY.pack(acc.data_ptr(), acc.stride(0), acc.stride(1), group, prev_len)


def _score_shape(plan, B: int, H: int) -> tuple:
    """Shape of the caller-supplied scores of a SCORE_GIVEN_SCORE(_SHARED) plan."""
    region = plan.sel_hi - plan.sel_lo
    return (B, region) if plan.score == P.SCORE_GIVEN_SCORE_SHARED else (B, H, region)
_lib = None
_WS_NEED = {}  # (plan set, group) -> workspace bytes the launch needs (0: everything fits on chip)


def library_path() -> str:
    return _LIB_PATH


def load_library():
    """Load the device library once; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"{_LIB_NAME} not found at {_LIB_PATH}: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a). kvcompress-b200 has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(_LIB_PATH)
    lib.kvc_abi_version.restype = ctypes.c_int
    lib.kvc_build_info.restype = ctypes.c_char_p
    lib.kvc_status_string.restype = ctypes.c_char_p
    lib.kvc_status_string.argtypes = [ctypes.c_int]
    lib.kvc_last_cuda_error.restype = ctypes.c_char_p
    lib.kvc_launch_count.restype = ctypes.c_int64
    lib.kvc_max_region_rows.restype = ctypes.c_int32
    lib.kvc_max_region_rows.argtypes = [ctypes.c_int32, ctypes.c_int32]
    lib.kvc_compress_layers.restype = ctypes.c_int
    lib.kvc_compress_layers.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_char_p,
                                        ctypes.c_void_p]
    lib.kvc_key_norms.restype = ctypes.c_int
    lib.kvc_key_norms.argtypes = [ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                  ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    lib.kvc_select.restype = ctypes.c_int
    lib.kvc_select.argtypes = [ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32,
                               ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p, ctypes.c_void_p]
    lib.kvc_slab_append.restype = ctypes.c_int
    lib.kvc_slab_append.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_void_p]
    lib.kvc_slab_compress.restype = ctypes.c_int
    lib.kvc_slab_compress.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_char_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64,
                                      ctypes.c_void_p]
    lib.kvc_workspace_bytes.restype = ctypes.c_int64
    lib.kvc_workspace_bytes.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p]
    lib.kvc_compress_layers_ws.restype = ctypes.c_int
    lib.kvc_compress_layers_ws.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_char_p,
                                           ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    lib.kvc_snapkv_vote.restype = ctypes.c_int
    lib.kvc_snapkv_vote.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32,
                                    ctypes.c_void_p]
    lib.kvc_snapkv_vote_compress.restype = ctypes.c_int
    lib.kvc_snapkv_vote_compress.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_char_p,
                                             ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_void_p]
    lib.kvc_h2o_accumulate.restype = ctypes.c_int
    lib.kvc_h2o_accumulate.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_float, ctypes.c_void_p]
    lib.kvc_h2o_qk_workspace_bytes.restype = ctypes.c_int64
    lib.kvc_h2o_qk_workspace_bytes.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_char_p]
    lib.kvc_h2o_accumulate_qk.restype = ctypes.c_int
    lib.kvc_h2o_accumulate_qk.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_int32, ctypes.c_char_p, ctypes.c_float,
                                          ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    lib.kvc_h2o_qk_tc_workspace_bytes.restype = ctypes.c_int64
    lib.kvc_h2o_qk_tc_workspace_bytes.argtypes = lib.kvc_h2o_qk_workspace_bytes.argtypes
    lib.kvc_h2o_accumulate_qk_tc.restype = ctypes.c_int
    lib.kvc_h2o_accumulate_qk_tc.argtypes = lib.kvc_h2o_accumulate_qk.argtypes
    lib.kvc_compress_layers_carry.restype = ctypes.c_int
    lib.kvc_compress_layers_carry.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_char_p,
                                              ctypes.c_char_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]
    lib.kvc_slab_compress_carry.restype = ctypes.c_int
    lib.kvc_slab_compress_carry.argtypes = [ctypes.c_char_p, ctypes.c_int32, ctypes.c_char_p, ctypes.c_char_p,
                                            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_char_p, ctypes.c_void_p,
                                            ctypes.c_int64, ctypes.c_void_p]
    if lib.kvc_abi_version() != KVC_ABI_VERSION:
        raise RuntimeError(f"{_LIB_NAME}: ABI version {lib.kvc_abi_version()} != {KVC_ABI_VERSION} — rebuild the library")
    _lib = lib
    return lib


_fast = None
_fast_tried = False
_KIND_CODE = {P.KEEP: 0, P.VIEW: 1, P.GATHER: 2}


def fast_binding():
    """The compiled per-call binding (csrc/kvc_fast_binding.cpp -> kvcompress/_kvc_fast*.so) or None when it has not
    been built.  It only replaces the per-layer pointer walk below with C++; the device library, the planner and
    every error message stay where they are, so without it the same calls simply cost more host time."""
    global _fast, _fast_tried
    if not _fast_tried:
        _fast_tried = True
        try:
            from . import _kvc_fast as mod

            _fast = mod if mod.KVC_ABI_VERSION == KVC_ABI_VERSION else None
        except ImportError:
            _fast = None
    return _fast


def launch_count() -> int:
    """Kernels launched by the library so far in this process."""
    return int(load_library().kvc_launch_count())


def _check(status: int, what: str) -> None:
    if status == KVC_OK:
        return
    lib = load_library()
    msg = lib.kvc_status_string(status).decode()
    if status == 4:
        msg += ": " + lib.kvc_last_cuda_error().decode()
    raise _STATUS_EXC.get(status, RuntimeError)(f"{what}: {msg}")


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{what}: tensor is on {t.device}; kvcompress-b200 runs on CUDA (sm_100a) only — there is no CPU path"
        )
    if t.dtype not in KVC_DTYPE:
        raise ValueError(f"{what}: dtype {t.dtype} is not supported (float32, float16, bfloat16)")


def _require_gpu_reachable(t: torch.Tensor, what: str) -> None:
    """CUDA tensors, or pinned host tensors (mapped into the device address space under UVA)."""
    if not t.is_cuda and not (t.device.type == "cpu" and t.is_pinned()):
        raise RuntimeError(
            f"{what}: tensor is on {t.device} in pageable memory; kvcompress-b200 runs on CUDA (sm_100a) only — "
            "there is no CPU path (pin host-resident caches with .pin_memory() to have the GPU compress them in place)"
        )
    if t.dtype not in KVC_DTYPE:
        raise ValueError(f"{what}: dtype {t.dtype} is not supported (float32, float16, bfloat16)")


def _rows_ok(t: torch.Tensor) -> bool:
    e = t.element_size()
    st = t.stride()
    return (st[3] == 1 or t.size(3) == 1) and (st[0] * e) % 16 == 0 and (st[1] * e) % 16 == 0 \
        and (st[2] * e) % 16 == 0 and t.data_ptr() % 16 == 0


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class PlanSet:
    """The per-layer plans of one call with everything the launch needs precomputed (which layers
    gather, which become views, the packed ``kvc_layer_plan`` records).  Built once per distinct
    (method arguments, sequence lengths) and cached by the method wrappers: a decode loop calls the
    same plan every step, so the per-step host work is pointers and one allocation."""

    __slots__ = ("plans", "gather", "views", "packed", "out_lens", "_fast")

    def __init__(self, plans: Sequence[P.LayerPlan]):
        self.plans = list(plans)
        self.gather = [i for i, p in enumerate(self.plans) if p.kind == P.GATHER]
        self.views = [(i, p.view_n) for i, p in enumerate(self.plans) if p.kind == P.VIEW]
        self.packed = {i: _PLAN.pack(p.seq_len, p.sink, p.sel_lo, p.sel_hi, p.k_sel, p.tail, p.score, p.pool_kernel)
                       for i, p in ((i, self.plans[i]) for i in self.gather)}
        self.out_lens = {i: self.plans[i].out_len for i in self.gather}
        self._fast = None

    def fast(self):
        """This plan set inside the compiled binding (built on first use), or None."""
        if self._fast is None:
            mod = fast_binding()
            if mod is None or not self.gather:
                self._fast = False
            else:
                lib = load_library()
                recs = [[_KIND_CODE[p.kind], p.seq_len, p.sink, p.sel_lo, p.sel_hi, p.k_sel, p.tail, p.score, p.pool_kernel]
                        for p in self.plans]
                self._fast = mod.FastPlans(recs, ctypes.cast(lib.kvc_compress_layers_ws, ctypes.c_void_p).value,
                                           ctypes.cast(lib.kvc_workspace_bytes, ctypes.c_void_p).value)
        return self._fast or None

    def __len__(self):
        return len(self.plans)

    def __getitem__(self, i):
        return self.plans[i]

    def __iter__(self):
        return iter(self.plans)


def run_plans(kv: Sequence[Tuple[torch.Tensor, torch.Tensor]], plans, given_indices: Optional[dict] = None,
              return_indices: bool = False, given_scores: Optional[dict] = None, norms: Optional[Sequence] = None,
              non_blocking: bool = False, output_device=None, carry: Optional[dict] = None):
    """Apply per-layer plans (a list of ``LayerPlan`` or a cached :class:`PlanSet`) to a list of (K, V) pairs.

    KEEP layers keep their tensor objects, VIEW layers become ``x[:, :, -n:, :]`` views (both
    exactly as the reference does); all GATHER layers of the call go to the device library in
    one ``kvc_compress_layers`` call per (device, dtype, B, H, D) group — normally one launch.
    The outputs of a group with one common length are carved out of ONE allocation.

    given_indices: {layer_idx: int32 tensor [B, H, k_sel]} for SCORE_GIVEN_INDEX plans.
    given_scores: {layer_idx: cache-dtype tensor [B, H, sel_hi - sel_lo]} for SCORE_GIVEN_SCORE plans,
        [B, sel_hi - sel_lo] (one row per batch entry, shared by its heads) for SCORE_GIVEN_SCORE_SHARED plans.
    return_indices: also return {layer_idx: int32 tensor [B, H, C]} of kept absolute rows.
    norms: per-layer stored key norms (``[B, H, >= S]``, cache dtype, last dim dense; ``None`` entries allowed) — what
        ``torch.norm(K, p=2, dim=-1)`` returns for the rows.  Layers that have them are ranked from 2-4 bytes per row
        instead of reading the K rows of the selection region (a :class:`KVSlabCache` records them at append time).
    non_blocking: host-resident (pinned) caches only — do not synchronise before returning; the pinned outputs are
        complete once the current stream has been synchronised.
    output_device: host-resident (pinned) caches only — a CUDA device that receives the compressed cache instead of
        pinned host memory (stream-ordered like any CUDA tensor: no synchronisation).
    carry: {layer_idx: (acc, group, prev_len)} — per-row state that follows the kept rows, in place and in the same
        launch (``kvc_compress_layers_carry``): ``acc[:, h*group+g, i] = acc[:, h*group+g, src(i)]`` for the kept rows
        ``src(i) < prev_len``, 0 for the others; acc is ``[B, H * group, >= S]`` in the cache dtype (H2O accumulators,
        :class:`~kvcompress.methods.h2o_attention.H2OScoreSlab` with ``carry_scores=True``).
    """
    ps = plans if isinstance(plans, PlanSet) else PlanSet(plans)
    if given_indices is None and given_scores is None and not return_indices and carry is None and ps.gather \
            and not ps.views:
        # the common per-step call: the compiled binding walks the layers (None: not built, or a case it leaves to us)
        fp = ps.fast()
        first = kv[ps.gather[0]][0] if len(kv) == len(ps.plans) else None
        if fp is not None and isinstance(first, torch.Tensor) and first.is_cuda:
            done = fp.run(kv if type(kv) is list else list(kv), norms)   # launches on torch's current stream
            if done is not None:
                return done
    out: List[Tuple[torch.Tensor, torch.Tensor]] = list(kv)
    for li, n in ps.views:
        keys, values = kv[li][0], kv[li][1]
        out[li] = (keys[:, :, -n:, :], values[:, :, -n:, :])
    indices = {}
    if not ps.gather:
        return (out, indices) if return_indices else out

    groups = {}
    for li in ps.gather:
        keys, values = kv[li][0], kv[li][1]
        _require_gpu_reachable(keys, f"layer {li} keys")
        _require_gpu_reachable(values, f"layer {li} values")
        shape = keys.shape
        if len(shape) != 4 or values.shape != shape or values.dtype != keys.dtype or values.device != keys.device:
            raise ValueError(f"layer {li}: keys/values must be matching [B, H, S, D] tensors")
        if shape[2] != ps.plans[li].seq_len:
            raise ValueError(f"layer {li}: plan built for seq_len {ps.plans[li].seq_len}, tensor has {shape[2]}")
        if (shape[3] * keys.element_size()) % 16 != 0:
            raise ValueError(f"layer {li}: head_dim*itemsize = {shape[3] * keys.element_size()} B is not a multiple of 16")
        groups.setdefault((keys.device, keys.dtype, shape[0], shape[1], shape[3]), []).append((li, keys, values))

    keepalive = []
    lib = load_library()
    for (device, dtype, B, H, D), members in groups.items():
        on_host = device.type == "cpu"
        if on_host and not torch.cuda.is_available():
            raise RuntimeError("pinned host tensors need a CUDA device to run on: there is no CPU path")
        run_device = torch.device("cuda", torch.cuda.current_device()) if on_host else device
        to_device = on_host and output_device is not None
        if to_device:
            run_device = torch.device(output_device)
            if run_device.type != "cuda":
                raise ValueError(f"output_device must be a CUDA device, got {run_device}")
            if run_device.index is None:
                run_device = torch.device("cuda", torch.cuda.current_device())
        alloc = dict(dtype=dtype, pin_memory=True) if on_host and not to_device else dict(dtype=dtype, device=run_device)
        n = len(members)
        lens = [ps.out_lens[li] for li, _, _ in members]
        C0 = lens[0]
        uniform = all(c == C0 for c in lens)
        # one allocation for every output of the group; per-layer tensors are views of it
        if uniform:
            big = torch.empty((2 * n, B, H, C0, D), **alloc)
            parts = big.unbind(0)
            base = big.data_ptr()
            step = B * H * C0 * D * big.element_size()
        else:  # per-layer budgets (pyramid_kv): one flat buffer split into [K0, V0, K1, V1, ...]
            sizes = [B * H * c * D for c in lens for _ in (0, 1)]
            flat = torch.empty((sum(sizes),), **alloc)
            chunks = flat.split_with_sizes(sizes)
            base = flat.data_ptr()
            esz = flat.element_size()
            offs = [0]
            for sz in sizes:
                offs.append(offs[-1] + sz * esz)
        plan_buf = bytearray(_PLAN.size * n)
        io_buf = bytearray(_IO.size * n)
        carry_buf = bytearray(_CARRY.size * n) if carry else None
        host_temps = False  # pinned temporaries made here: they must outlive the launch that reads them
        for m, (li, keys, values) in enumerate(members):
            plan = ps.plans[li]
            if not _rows_ok(keys):
                keys = keys.contiguous().pin_memory() if on_host else keys.contiguous()
                keepalive.append(keys)
                host_temps = host_temps or on_host
            if not _rows_ok(values):
                values = values.contiguous().pin_memory() if on_host else values.contiguous()
                keepalive.append(values)
                host_temps = host_temps or on_host
            if uniform:
                k_out, v_out = parts[2 * m], parts[2 * m + 1]
                k_out_ptr, v_out_ptr = base + 2 * m * step, base + (2 * m + 1) * step
            else:
                k_out = chunks[2 * m].view(B, H, lens[m], D)
                v_out = chunks[2 * m + 1].view(B, H, lens[m], D)
                k_out_ptr, v_out_ptr = base + offs[2 * m], base + offs[2 * m + 1]
            out[li] = (k_out, v_out)
            idx_out_ptr = 0
            if return_indices:
                idx = torch.empty((B, H, lens[m]), **dict(alloc, dtype=torch.int32))
                indices[li] = idx
                idx_out_ptr = idx.data_ptr()
            idx_in_ptr = 0
            if plan.score == P.SCORE_GIVEN_INDEX and plan.k_sel > 0:
                gi = None if given_indices is None else given_indices.get(li)
                if gi is None:
                    raise ValueError(f"layer {li}: plan needs caller-supplied indices")
                if gi.dtype != torch.int32 or not gi.is_contiguous() or tuple(gi.shape) != (B, H, plan.k_sel) \
                        or gi.device != device:
                    raise ValueError(f"layer {li}: indices must be a contiguous int32 [B, H, k_sel] tensor on {device}")
                if on_host and not gi.is_pinned():
                    gi = gi.pin_memory()
                    host_temps = True
                idx_in_ptr = gi.data_ptr()
                keepalive.append(gi)
            score_in_ptr = 0
            if plan.score in _GIVEN_SCORES and plan.k_sel > 0:
                gs = None if given_scores is None else given_scores.get(li)
                if gs is None:
                    raise ValueError(f"layer {li}: plan needs caller-supplied scores")
                want = _score_shape(plan, B, H)
                if gs.dtype != dtype or not gs.is_contiguous() or tuple(gs.shape) != want or gs.device != device:
                    raise ValueError(f"layer {li}: scores must be a contiguous {dtype} {list(want)} tensor on {device}")
                if on_host and not gs.is_pinned():
                    gs = gs.pin_memory()
                    host_temps = True
                score_in_ptr = gs.data_ptr()
                keepalive.append(gs)
            norms_ptr, nsb, nsh = 0, 0, 0
            nt = None if norms is None else norms[li]
            if nt is not None and plan.k_sel > 0 and plan.score in _RANKED:
                if nt.dtype != dtype or nt.dim() != 3 or nt.size(0) != B or nt.size(1) != H or nt.size(2) < plan.seq_len \
                        or nt.stride(2) != 1 or nt.device != device:
                    raise ValueError(f"layer {li}: stored norms must be a {dtype} [B, H, >= S] tensor on {device} "
                                     "with a dense last dimension")
                if on_host and not nt.is_pinned():
                    raise RuntimeError(f"layer {li}: stored norms of a host-resident cache must be pinned")
                norms_ptr, nsb, nsh = nt.data_ptr(), nt.stride(0), nt.stride(1)
                keepalive.append(nt)
            if carry_buf is not None and carry.get(li) is not None:
                carry_buf[m * _CARRY.size:(m + 1) * _CARRY.size] = carry_record(li, carry[li], B, H, dtype, plan.seq_len)
            plan_buf[m * _PLAN.size:(m + 1) * _PLAN.size] = ps.packed[li]
            ks, vs = keys.stride(), values.stride()
            _IO.pack_into(io_buf, m * _IO.size, keys.data_ptr(), values.data_ptr(), k_out_ptr, v_out_ptr,
                          ks[0], ks[1], ks[2], vs[0], vs[1], vs[2], idx_out_ptr, idx_in_ptr, score_in_ptr,
                          norms_ptr, nsb, nsh)
        dev_index = run_device.index if run_device.index is not None else torch.cuda.current_device()
        shape_rec = _SHAPE.pack(B, H, D, KVC_DTYPE[dtype], dev_index)
        plan_bytes = bytes(plan_buf)
        ws_key = (id(ps), B, H, D, dtype, tuple(li for li, _, _ in members))
        need = _WS_NEED.get(ws_key)
        if need is None or need[0] is not ps:
            need = (ps, int(lib.kvc_workspace_bytes(shape_rec, n, plan_bytes)))
            if len(_WS_NEED) > 256:
                _WS_NEED.clear()
            _WS_NEED[ws_key] = need
        ws_ptr, ws_bytes = None, 0
        if need[1] > 0:  # selection larger than shared memory: radix keys / kept indices in a device workspace
            ws = torch.empty((need[1],), dtype=torch.uint8, device=run_device)
            keepalive.append(ws)
            ws_ptr, ws_bytes = ctypes.c_void_p(ws.data_ptr()), need[1]
        # a NULL carry is exactly kvc_compress_layers_ws (kvc.h)
        status = lib.kvc_compress_layers_carry(shape_rec, n, plan_bytes, bytes(io_buf),
                                               None if carry_buf is None else bytes(carry_buf), ws_ptr, ws_bytes,
                                               ctypes.c_void_p(_stream_ptr(run_device)))
        _check(status, "kvc_compress_layers")
        if on_host and (host_temps or not (non_blocking or to_device)):
            # host tensors are read by the caller with plain loads: finish before returning, as the reference's
            # (synchronous) CPU path does; non_blocking=True leaves that to the caller (tensor.to(..., non_blocking=True)).
            # Pinned temporaries (re-laid-out inputs, re-pinned indices) are not stream-ordered like device memory: the
            # launch that reads them has to finish before they go back to the host allocator.
            torch.cuda.current_stream(run_device).synchronize()
    if return_indices:
        return out, indices
    return out


def key_norms(keys: torch.Tensor, row_lo: int = 0, row_hi: Optional[int] = None) -> torch.Tensor:
    """``torch.norm(keys[:, :, row_lo:row_hi], p=2, dim=-1)`` on the device library (K1)."""
    _require_cuda(keys, "keys")
    if keys.dim() != 4:
        raise ValueError("keys must be [B, H, S, D]")
    if not _rows_ok(keys):
        keys = keys.contiguous()
    B, H, S, D = keys.shape
    row_hi = S if row_hi is None else row_hi
    out = torch.empty((B, H, max(row_hi - row_lo, 0)), dtype=keys.dtype, device=keys.device)
    shape = _SHAPE.pack(B, H, D, KVC_DTYPE[keys.dtype], keys.device.index)
    status = load_library().kvc_key_norms(shape, keys.data_ptr(), keys.stride(0), keys.stride(1), keys.stride(2),
                                          row_lo, row_hi, out.data_ptr(), ctypes.c_void_p(_stream_ptr(keys.device)))
    _check(status, "kvc_key_norms")
    return out


def select(scores: torch.Tensor, k: int, largest: bool = False) -> torch.Tensor:
    """Ascending indices of the k smallest (largest) scores per row, ties to the lowest index (K2)."""
    _require_cuda(scores, "scores")
    scores = scores.contiguous()
    n = scores.size(-1)
    rows = scores.numel() // max(n, 1)
    out = torch.empty(tuple(scores.shape[:-1]) + (k,), dtype=torch.int32, device=scores.device)
    status = load_library().kvc_select(KVC_DTYPE[scores.dtype], scores.device.index, scores.data_ptr(), rows, n, k,
                                       1 if largest else 0, out.data_ptr(),
                                       ctypes.c_void_p(_stream_ptr(scores.device)))
    _check(status, "kvc_select")
    return out


_VOTE = struct.Struct("3P6q2iP")  # kvc_vote_layer: k_in q_obs votes_out | 6 strides | seq_len reserved | lse
assert _VOTE.size == 88


def _vote_records(layers: Sequence[Tuple[torch.Tensor, torch.Tensor]], window: int, lse: Optional[Sequence]):
    """Validate (keys, obs_queries[, lse]) per layer and pack the ``kvc_vote_layer`` records.
    Returns (shape record, packed records, votes tensors, group size, keep-alive list, prepared keys)."""
    k0, q0 = layers[0]
    _require_cuda(k0, "keys")
    B, H, _, D = k0.shape
    if q0.dim() != 4 or q0.size(0) != B or q0.size(1) % H or q0.size(2) != window or q0.size(3) != D:
        raise ValueError(f"obs_queries must be [B={B}, H*G, W={window}, D={D}], got {tuple(q0.shape)}")
    G = q0.size(1) // H
    if k0.dtype not in (torch.bfloat16, torch.float16):
        raise ValueError("the q.K^T vote runs on bfloat16/float16 caches")
    if D * 2 // 16 not in (8, 10, 16) or (D * 2) % 16:
        raise ValueError(f"head_dim {D}: the vote kernel covers head_dim 64, 80 and 128")
    if G * window > 128:
        raise ValueError(f"group size x observation_window = {G * window} exceeds the 128 query rows of one MMA")
    if lse is not None and len(lse) != len(layers):
        raise ValueError(f"obs_lse: {len(lse)} entries for {len(layers)} layers")
    out, keep, prepared = [], [], []
    buf = bytearray(_VOTE.size * len(layers))
    for m, (keys, q) in enumerate(layers):
        _require_cuda(keys, f"layer {m} keys")
        _require_cuda(q, f"layer {m} obs_queries")
        if keys.shape[:2] != (B, H) or keys.size(3) != D or keys.dtype != k0.dtype or q.dtype != k0.dtype \
                or tuple(q.shape) != tuple(q0.shape) or keys.device != k0.device or q.device != k0.device:
            raise ValueError(f"layer {m}: keys / obs_queries do not match layer 0's shape, dtype or device")
        if keys.size(2) <= window:
            raise ValueError(f"layer {m}: {keys.size(2)} rows do not exceed the observation window {window}")
        if not _rows_ok(keys):
            keys = keys.contiguous()
        if not _rows_ok(q):
            q = q.contiguous()
        lse_ptr = 0
        if lse is not None and lse[m] is not None:
            t = lse[m]
            if t.dtype != torch.float32 or tuple(t.shape) != (B, H * G, window) or t.device != k0.device:
                raise ValueError(f"layer {m}: obs_lse must be a float32 [B={B}, H*G={H * G}, W={window}] tensor on {k0.device}")
            t = t.contiguous()
            keep.append(t)
            lse_ptr = t.data_ptr()
        keep.append((keys, q))
        prepared.append(keys)
        votes = torch.empty((B, H, keys.size(2) - window), dtype=keys.dtype, device=keys.device)
        out.append(votes)
        ks, qs = keys.stride(), q.stride()
        _VOTE.pack_into(buf, m * _VOTE.size, keys.data_ptr(), q.data_ptr(), votes.data_ptr(), ks[0], ks[1], ks[2],
                        qs[0], qs[1], qs[2], keys.size(2), 0, lse_ptr)
    shape = _SHAPE.pack(B, H, D, KVC_DTYPE[k0.dtype], k0.device.index)
    return shape, bytes(buf), out, G, keep, prepared


def snapkv_votes(layers: Sequence[Tuple[torch.Tensor, torch.Tensor]], window: int,
                 lse: Optional[Sequence[Optional[torch.Tensor]]] = None) -> List[torch.Tensor]:
    """Observation-window votes on the tensor cores (tcgen05), one launch for every (keys, obs_queries) pair.

    layers: [(keys [B,H,S,D], obs_queries [B,H*G,W,D]), ...] 16-bit CUDA tensors of one shape.
    lse: optional per-layer ``[B, H*G, W]`` float32 log-sum-exp of the window queries' attention rows (what a
        flash-attention forward returns): the kernel then reads K once instead of twice.
    Returns votes [B,H,S-W] per layer (cache dtype):
    ``softmax(Q K^T / sqrt(D), causal inside the window)[..., :S-W].sum over the window queries and the group``."""
    if not layers:
        return []
    shape, recs, out, G, keep, _ = _vote_records(layers, window, lse)
    k0 = layers[0][0]
    status = load_library().kvc_snapkv_vote(shape, len(layers), recs, G, window, ctypes.c_void_p(_stream_ptr(k0.device)))
    _check(status, "kvc_snapkv_vote")
    return out


def snapkv_vote_compress(kv: Sequence[Tuple[torch.Tensor, torch.Tensor]], plans, obs_queries: Sequence, window: int,
                         lse: Optional[Sequence] = None, return_indices: bool = False, return_votes: bool = False):
    """snapkv_lite in vote mode, ONE launch: per (layer, b, h) the vote, ``avg_pool1d``, top-k, sort and the K/V gather
    (reference snapkv_lite.py:104-150 behind the q.K^T vote).  ``plans``: the snapkv plans with
    ``SCORE_GIVEN_SCORE`` on the layers that vote; other layers follow their plan as in :func:`run_plans`.
    Prefixes too long for the kernel's shared memory run as vote launch + select/gather launch instead."""
    ps = plans if isinstance(plans, PlanSet) else PlanSet(plans)
    voted = [li for li in ps.gather if ps.plans[li].score == P.SCORE_GIVEN_SCORE and ps.plans[li].k_sel > 0]
    rest = [li for li in ps.gather if li not in voted]
    out: List[Tuple[torch.Tensor, torch.Tensor]] = list(kv)
    indices, votes_by_layer = {}, {}
    if rest or ps.views:  # layers that do not vote (tail-only budgets): the ordinary path
        other = [p if li not in voted else P.LayerPlan(P.KEEP, p.seq_len) for li, p in enumerate(ps.plans)]
        res = run_plans(kv, other, return_indices=return_indices)
        out, idx = res if return_indices else (res, {})
        indices.update(idx)
    if voted:
        shape, recs, votes, G, keep, keys_used = _vote_records([(kv[li][0], obs_queries[li]) for li in voted], window,
                                                               None if lse is None else [lse[li] for li in voted])
        k0 = kv[voted[0]][0]
        B, H, _, D = k0.shape
        plan_buf = bytearray(_PLAN.size * len(voted))
        io_buf = bytearray(_IO.size * len(voted))
        lens = [ps.out_lens[li] for li in voted]
        sizes = [B * H * c * D for c in lens for _ in (0, 1)]
        flat = torch.empty((sum(sizes),), dtype=k0.dtype, device=k0.device)
        chunks = flat.split_with_sizes(sizes)
        for m, li in enumerate(voted):
            keys, values = keys_used[m], kv[li][1]
            _require_cuda(values, f"layer {li} values")
            if values.shape != kv[li][0].shape or values.dtype != keys.dtype or values.device != keys.device:
                raise ValueError(f"layer {li}: keys/values must be matching [B, H, S, D] tensors")
            if not _rows_ok(values):
                values = values.contiguous()
                keep.append(values)
            k_out, v_out = chunks[2 * m].view(B, H, lens[m], D), chunks[2 * m + 1].view(B, H, lens[m], D)
            out[li] = (k_out, v_out)
            idx_ptr = 0
            if return_indices:
                indices[li] = torch.empty((B, H, lens[m]), dtype=torch.int32, device=keys.device)
                idx_ptr = indices[li].data_ptr()
            plan_buf[m * _PLAN.size:(m + 1) * _PLAN.size] = ps.packed[li]
            ks, vs = keys.stride(), values.stride()
            _IO.pack_into(io_buf, m * _IO.size, keys.data_ptr(), values.data_ptr(), k_out.data_ptr(), v_out.data_ptr(),
                          ks[0], ks[1], ks[2], vs[0], vs[1], vs[2], idx_ptr, 0, 0, 0, 0, 0)
            votes_by_layer[li] = votes[m]
        lib = load_library()
        status = lib.kvc_snapkv_vote_compress(shape, len(voted), recs, bytes(plan_buf), bytes(io_buf), G, window,
                                              ctypes.c_void_p(_stream_ptr(k0.device)))
        if status == 3:  # prefix too long for the fused tail: votes, then select + gather with a workspace
            status = lib.kvc_snapkv_vote(shape, len(voted), recs, G, window, ctypes.c_void_p(_stream_ptr(k0.device)))
            _check(status, "kvc_snapkv_vote")
            two = [p if li in voted else P.LayerPlan(P.KEEP, p.seq_len) for li, p in enumerate(ps.plans)]
            res = run_plans(kv, two, given_scores=votes_by_layer, return_indices=return_indices)
            res, idx = res if return_indices else (res, {})
            for li in voted:
                out[li] = res[li]
            indices.update(idx)
        else:
            _check(status, "kvc_snapkv_vote_compress")
    ret = [out]
    if return_indices:
        ret.append(indices)
    if return_votes:
        ret.append(votes_by_layer)
    return ret[0] if len(ret) == 1 else tuple(ret)


_H2O = struct.Struct("P3qP2qP6i")  # kvc_h2o_layer: attn | 3 strides | acc | 2 strides | score_out | n_query key_len prev_len
assert _H2O.size == 88             #                score_lo score_hi reserved


def h2o_accumulate(layers: Sequence[tuple], decay: float) -> None:
    """H2O attention-score bookkeeping for several layers in ONE ``kvc_h2o_accumulate`` launch.

    layers: ``(attn, acc, score_out, prev_len, key_len, score_lo, score_hi)`` per layer —
      attn ``[B, Hq, n_query, key_len]`` attention probabilities with a dense last dimension, or ``None`` to only
      re-score; acc ``[B, Hq, >= key_len]`` accumulators (same dtype, dense last dimension), updated in place:
      ``acc = round(round(acc * decay) + attn.sum(dim=2))`` for ``j < prev_len``, ``attn.sum(dim=2)`` beyond it (from
      zero when ``prev_len < 0`` or ``> key_len``); score_out ``[>= B * (score_hi - score_lo)]`` dense, or ``None``:
      ``acc[:, :, score_lo:score_hi].sum(dim=1)`` of the updated accumulators.
    Every tensor must be a CUDA tensor of one dtype and device, with one (B, Hq); nothing is synchronised."""
    if not layers:
        return
    acc0 = layers[0][1]
    _require_cuda(acc0, "acc")
    B, Hq = acc0.size(0), acc0.size(1)
    buf = bytearray(_H2O.size * len(layers))
    for m, (attn, acc, score, prev_len, key_len, lo, hi) in enumerate(layers):
        if acc.dtype != acc0.dtype or acc.device != acc0.device or acc.dim() != 3 or acc.size(0) != B \
                or acc.size(1) != Hq or acc.size(2) < key_len or acc.stride(2) != 1:
            raise ValueError(f"layer {m}: acc must be a [B={B}, Hq={Hq}, >= {key_len}] {acc0.dtype} tensor on "
                             f"{acc0.device} with a dense last dimension")
        a_ptr, a_st, n_query = 0, (0, 0, 0), 0
        if attn is not None:
            _require_cuda(attn, f"layer {m} attention")
            if attn.dtype != acc0.dtype or attn.device != acc0.device or attn.dim() != 4 or attn.size(0) != B \
                    or attn.size(1) != Hq or attn.size(3) != key_len or (attn.stride(3) != 1 and key_len > 1):
                raise ValueError(f"layer {m}: attention must be a [B={B}, Hq={Hq}, n_query, {key_len}] {acc0.dtype} "
                                 f"tensor on {acc0.device} with a dense last dimension")
            a_ptr, a_st, n_query = attn.data_ptr(), attn.stride()[:3], attn.size(2)
        s_ptr = 0
        if score is not None:
            if score.dtype != acc0.dtype or score.device != acc0.device or not score.is_contiguous() \
                    or score.numel() < B * (hi - lo):
                raise ValueError(f"layer {m}: score_out must be a contiguous {acc0.dtype} tensor of >= B * region "
                                 f"elements on {acc0.device}")
            s_ptr = score.data_ptr()
        _H2O.pack_into(buf, m * _H2O.size, a_ptr, a_st[0], a_st[1], a_st[2], acc.data_ptr(), acc.stride(0),
                       acc.stride(1), s_ptr, n_query, key_len, prev_len, lo, hi, 0)
    shape = _SHAPE.pack(B, Hq, 0, KVC_DTYPE[acc0.dtype], acc0.device.index)
    status = load_library().kvc_h2o_accumulate(shape, len(layers), bytes(buf), float(decay),
                                               ctypes.c_void_p(_stream_ptr(acc0.device)))
    _check(status, "kvc_h2o_accumulate")


_H2O_QK = struct.Struct("P3qP3qP2qP2qPf5i")  # kvc_h2o_qk_layer: q | 3 strides | k | 3 strides | mask | 2 strides | acc |
assert _H2O_QK.size == 144                    # 2 strides | score_out | scaling | n_query key_len prev_len score_lo score_hi


def h2o_accumulate_qk(layers: Sequence[tuple], decay: float, group: int, workspace, tensor_cores: bool = False) -> None:
    """H2O attention-score bookkeeping from queries and keys (``kvc_h2o_accumulate_qk``): two launches for all layers.

    layers: ``(q, k, mask, acc, score_out, prev_len, score_lo, score_hi, scaling)`` per layer —
      q ``[B, Hq, T, D]`` post-RoPE queries with a dense last dimension, Hq = group * Hkv; k ``[B, Hkv, key_len, D]`` keys
      whose rows are 16-byte aligned (any slab view); mask ``[B, T, >= key_len]`` bool (True = visible) with a dense last
      dimension, or ``None`` for the causal rule (query t sees keys ``j <= key_len - T + t``); acc, score_out, prev_len,
      score_lo, score_hi as in :func:`h2o_accumulate`; scaling the logit scale (``D ** -0.5`` for most models).
      The probabilities are ``round(exp(s - lse))`` of the fp32 logits ``s = scaling * q . k`` where visible, 0 elsewhere.
    workspace: a uint8 CUDA tensor, or a callable that returns one of at least the bytes it is given.
    q, k and acc share one dtype and device; nothing is synchronised."""
    if not layers:
        return
    group = int(group)
    if group < 1:
        raise ValueError(f"group must be >= 1, got {group}")
    q0, k0, acc0 = layers[0][0], layers[0][1], layers[0][3]
    _require_cuda(k0, "keys")
    if k0.dim() != 4:
        raise ValueError(f"keys must be [B, Hkv, key_len, D], got {tuple(k0.shape)}")
    B, Hkv, _, D = k0.shape
    Hq = Hkv * group
    dt, dev = k0.dtype, k0.device
    buf = bytearray(_H2O_QK.size * len(layers))
    keep = []
    for m, (q, k, mask, acc, score, prev_len, lo, hi, scaling) in enumerate(layers):
        _require_cuda(q, f"layer {m} queries")
        _require_cuda(k, f"layer {m} keys")
        if k.dtype != dt or k.device != dev or k.dim() != 4 or k.shape[:2] != (B, Hkv) or k.size(3) != D:
            raise ValueError(f"layer {m}: keys must be a [B={B}, Hkv={Hkv}, key_len, D={D}] {dt} tensor on {dev}")
        key_len = k.size(2)
        if q.dtype != dt or q.device != dev or q.dim() != 4 or q.size(0) != B or q.size(1) != Hq or q.size(3) != D \
                or (q.stride(3) != 1 and D > 1):
            raise ValueError(f"layer {m}: queries must be a [B={B}, Hq={Hq}, T, D={D}] {dt} tensor on {dev} with a dense "
                             "last dimension")
        T = q.size(2)
        if acc.dtype != dt or acc.device != dev or acc.dim() != 3 or acc.size(0) != B or acc.size(1) != Hq \
                or acc.size(2) < key_len or acc.stride(2) != 1:
            raise ValueError(f"layer {m}: acc must be a [B={B}, Hq={Hq}, >= {key_len}] {dt} tensor on {dev} with a dense "
                             "last dimension")
        if not _rows_ok(k):
            k = k.contiguous()
            keep.append(k)
        if tensor_cores and not _rows_ok(q):  # a tensor map needs 16-byte aligned strides, size-1 dimensions included
            q = q.clone(memory_format=torch.contiguous_format)
            keep.append(q)
        m_ptr, m_st = 0, (0, 0)
        if mask is not None:
            if mask.dtype != torch.bool or mask.device != dev or mask.dim() != 3 or mask.size(0) != B \
                    or mask.size(1) != T or mask.size(2) < key_len or (mask.stride(2) != 1 and key_len > 1):
                raise ValueError(f"layer {m}: mask must be a bool [B={B}, T={T}, >= {key_len}] tensor on {dev} with a "
                                 "dense last dimension")
            m_ptr, m_st = mask.data_ptr(), mask.stride()[:2]
        elif T > key_len:
            raise ValueError(f"layer {m}: {T} queries over {key_len} keys need a mask")
        s_ptr = 0
        if score is not None:
            if score.dtype != dt or score.device != dev or not score.is_contiguous() or score.numel() < B * (hi - lo):
                raise ValueError(f"layer {m}: score_out must be a contiguous {dt} tensor of >= B * region elements on "
                                 f"{dev}")
            s_ptr = score.data_ptr()
        qs, ks = q.stride(), k.stride()
        _H2O_QK.pack_into(buf, m * _H2O_QK.size, q.data_ptr(), qs[0], qs[1], qs[2], k.data_ptr(), ks[0], ks[1], ks[2],
                          m_ptr, m_st[0], m_st[1], acc.data_ptr(), acc.stride(0), acc.stride(1), s_ptr, float(scaling),
                          T, key_len, prev_len, lo, hi)
    recs = bytes(buf)
    shape = _SHAPE.pack(B, Hkv, D, KVC_DTYPE[dt], dev.index)
    lib = load_library()
    name = "kvc_h2o_accumulate_qk_tc" if tensor_cores else "kvc_h2o_accumulate_qk"
    run = getattr(lib, name)
    sizer = lib.kvc_h2o_qk_tc_workspace_bytes if tensor_cores else lib.kvc_h2o_qk_workspace_bytes
    need = int(sizer(shape, group, len(layers), recs))
    if need < 0:
        status = run(shape, group, len(layers), recs, float(decay), None, 0, None)
        _check(status, name)
        raise ValueError(f"{name}: invalid arguments")
    ws = workspace(need) if callable(workspace) else workspace
    ws_ptr, ws_bytes = 0, 0
    if ws is not None:
        if ws.device != dev or not ws.is_contiguous():
            raise ValueError(f"workspace must be a contiguous tensor on {dev}")
        ws_ptr, ws_bytes = ws.data_ptr(), ws.numel() * ws.element_size()
    if ws_bytes < need:
        raise ValueError(f"workspace of {ws_bytes} bytes, {name} needs {need}")
    status = run(shape, group, len(layers), recs, float(decay), ctypes.c_void_p(ws_ptr), ws_bytes,
                 ctypes.c_void_p(_stream_ptr(dev)))
    _check(status, name)


def h2o_accumulate_qk_tc(layers: Sequence[tuple], decay: float, group: int, workspace) -> None:
    """:func:`h2o_accumulate_qk` on the tensor cores (``kvc_h2o_accumulate_qk_tc``): the same records and workspace
    callback, logits from ``tcgen05.mma`` (16-bit q and K, fp32 accumulation) and ``p = round(exp2(a * c - lse2))``,
    ``c = scaling * log2(e)``; the query sum, the decay update and the head sum are the CUDA-core form's.  bf16 / f16
    only, head_dim 64, 80 or 128, q and K with 16-byte aligned base and strides (``ValueError`` otherwise).  Two launches
    for every 32 layers, plus one for the score rows."""
    h2o_accumulate_qk(layers, decay, group, workspace, tensor_cores=True)
