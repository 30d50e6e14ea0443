"""kvcompress (B200-native): the per-step KV-cache compression hot path on sm_100a.

Drop-in for the compress surface of od-liu/CS3602-LLM-Inference-Acceleration's ``kvcompress``
(reference kvcompress/__init__.py:33-97): the same function names, signatures, defaults and
``[B, H, S, D]`` per-layer ``(K, V)`` layout, each call served by hand-written CUDA kernels in
``csrc/`` through the C ABI of ``include/kvc.h``.  All eight hot-path functions are exported at
top level (the reference exports three here and the rest under ``kvcompress.methods``).

There is no CPU path: tensors that need to be moved must be CUDA tensors.
"""

from .methods import (
    l2_compress,
    fix_size_l2_compress,
    streaming_llm_compress,
    evict_for_space,
    recent_only_compress,
    h2o_l2_compress,
    h2o_attention_compress,
    H2OAttentionManager,
    H2OScoreSlab,
    create_h2o_manager_from_model,
    snapkv_lite_compress,
    pyramid_kv_compress,
    adaptive_l2_compress,
    get_compress_fn,
    list_methods,
    register_method,
    COMPRESS_METHODS,
)
from .slab_cache import KVSlabCache
from .capture import capture_queries, QueryCapture
from .evaluate import evaluate_with_compression, evaluate_baseline, compare_methods
from .benchmark import benchmark, measure_generation_metrics, run_benchmark_suite, print_benchmark_summary
from .utils import (
    to_dynamic_cache,
    normalize_kv_cache,
    get_cache_size_mb,
    get_cache_info,
    get_seq_len,
)

__all__ = [
    "l2_compress", "fix_size_l2_compress", "streaming_llm_compress", "evict_for_space", "recent_only_compress",
    "h2o_l2_compress", "h2o_attention_compress", "H2OAttentionManager", "H2OScoreSlab",
    "create_h2o_manager_from_model",
    "snapkv_lite_compress", "pyramid_kv_compress", "adaptive_l2_compress",
    "get_compress_fn", "list_methods", "register_method", "COMPRESS_METHODS",
    "to_dynamic_cache", "normalize_kv_cache", "get_cache_size_mb", "get_cache_info", "get_seq_len",
    "evaluate_with_compression", "evaluate_baseline", "compare_methods",
    "benchmark", "measure_generation_metrics", "run_benchmark_suite", "print_benchmark_summary",
    "KVSlabCache", "capture_queries", "QueryCapture",
]

__version__ = "2.0.0"
