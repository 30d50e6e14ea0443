"""Registry of compression methods — the drop-in plugin surface (reference methods/__init__.py:21-78).

Every entry is a callable ``fn(past_key_values, <method kwargs>, skip_layers=..., **kwargs)`` returning a new list of
per-layer ``(K, V)`` tuples; all of them plan on the host and run one fused sm_100a launch per call."""

from importlib import import_module
from typing import Callable, Dict, List

# registry name, defining module, function name — in the order list_methods() reports (reference :21-33)
_METHOD_TABLE = (
    ("l2_compress", "l2_compress", "l2_compress"),
    ("fix_size_l2", "fix_size_l2", "fix_size_l2_compress"),
    ("streaming_llm", "streaming_llm", "streaming_llm_compress"),
    ("recent_only", "recent_only", "recent_only_compress"),
    ("h2o_l2", "h2o_l2", "h2o_l2_compress"),
    ("h2o_attention", "h2o_attention", "h2o_attention_compress"),
    ("snapkv_lite", "snapkv_lite", "snapkv_lite_compress"),
    ("pyramid_kv", "pyramid_kv", "pyramid_kv_compress"),
    ("adaptive_l2", "adaptive_l2", "adaptive_l2_compress"),
)
# helpers the reference exports next to the compress functions
_EXTRA_EXPORTS = (
    ("streaming_llm", "evict_for_space"),
    ("h2o_attention", "H2OAttentionManager"),
    ("h2o_attention", "H2OScoreSlab"),
    ("h2o_attention", "create_h2o_manager_from_model"),
)

COMPRESS_METHODS: Dict[str, Callable] = {}
__all__ = ["get_compress_fn", "list_methods", "register_method", "COMPRESS_METHODS"]

for _name, _module, _attr in _METHOD_TABLE:
    _fn = getattr(import_module(f"{__name__}.{_module}"), _attr)
    COMPRESS_METHODS[_name] = _fn
    globals()[_attr] = _fn
    __all__.append(_attr)
for _module, _attr in _EXTRA_EXPORTS:
    globals()[_attr] = getattr(import_module(f"{__name__}.{_module}"), _attr)
    __all__.append(_attr)
del _name, _module, _attr, _fn


def get_compress_fn(method: str) -> Callable:
    """The callable registered under ``method``; an unknown name raises ``ValueError`` naming what exists (:36-61)."""
    try:
        return COMPRESS_METHODS[method]
    except KeyError:
        raise ValueError(f"Unknown method: {method}. Available: {list(COMPRESS_METHODS)}") from None


def list_methods() -> List[str]:
    """Registered names, registration order (:64-66)."""
    return list(COMPRESS_METHODS)


def register_method(name: str, fn: Callable) -> None:
    """Add or replace ``name``; ``fn(past_key_values, **kwargs) -> List[Tuple[Tensor, Tensor]]`` (:69-78)."""
    COMPRESS_METHODS[name] = fn
