"""Oracle and host planner against the REAL reference, live, on randomly drawn calls.

The committed fixtures (tests/golden/) pin the oracle on 125 hand-picked cases.  Where a checkout of the original
project is named by the ``KVCOMPRESS_REFERENCE`` environment variable (the directory that holds its ``kvcompress``
package; it is not part of this repository, and nothing marked ``gpu`` reads it) this module additionally imports the
unmodified reference under a private module name and compares, for seeded random methods / arguments / shapes /
dtypes: output lengths, which layers come back untouched or as views, and the kept rows (identical on continuous fp32
data, valid under the tie rule on bf16 and on tie-heavy data).  Skipped without the checkout.
"""

import importlib.util
import os
import sys

import numpy as np
import pytest
import torch

import cases
from oracle import kvc_oracle as O
from test_planner import plan_for

REF_ROOT = os.environ.get("KVCOMPRESS_REFERENCE", "")
REF_DIR = os.path.join(os.path.abspath(REF_ROOT), "kvcompress") if REF_ROOT else ""
pytestmark = pytest.mark.skipif(not REF_DIR or not os.path.isfile(os.path.join(REF_DIR, "__init__.py")),
                                reason="KVCOMPRESS_REFERENCE does not name a checkout of the original project")


@pytest.fixture(scope="module")
def ref():
    """The reference package under the name ``kvcompress_ref_live`` (``kvcompress`` is this repo's package here)."""
    name = "kvcompress_ref_live"
    if name in sys.modules:
        return sys.modules[name]
    spec = importlib.util.spec_from_file_location(name, os.path.join(REF_DIR, "__init__.py"),
                                                  submodule_search_locations=[REF_DIR])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    dont = sys.dont_write_bytecode
    sys.dont_write_bytecode = True      # the checkout is read-only
    try:
        spec.loader.exec_module(mod)
    except BaseException:
        sys.modules.pop(name, None)
        raise
    finally:
        sys.dont_write_bytecode = dont
    assert mod.__file__.startswith(REF_DIR)
    return mod


def to_torch(a: np.ndarray, dtype: str) -> torch.Tensor:
    if dtype == "bf16":
        return torch.from_numpy(a.view(np.int16).copy()).view(torch.bfloat16)
    return torch.from_numpy(a.copy())


def draw_call(rng):
    """One random call: (method, kwargs, seq_lens, B, H, D, dtype, style)."""
    method = str(rng.choice(["l2_compress", "fix_size_l2", "streaming_llm", "recent_only", "h2o_l2", "snapkv_lite",
                             "pyramid_kv", "adaptive_l2"]))
    L = int(rng.integers(1, 5))
    base = int(rng.integers(1, 700))
    seq_lens = [base] * L if rng.random() < 0.7 else [int(rng.integers(1, 700)) for _ in range(L)]
    skip = sorted(set(int(x) for x in rng.integers(0, L, size=int(rng.integers(0, 3)))))
    cap = int(rng.integers(1, 400))
    if method == "l2_compress":
        kw = dict(keep_ratio=float(rng.choice([1.0, 0.9, 0.8, 0.5, 0.3, 0.05, round(float(rng.random()), 3) or 0.5])),
                  prune_after=int(rng.integers(0, 500)))
    elif method == "fix_size_l2":
        kw = dict(fix_kv_size=cap, keep_ratio=float(rng.choice([0.0, 0.2, 0.5, 0.9, 1.0, round(float(rng.random()), 3)])),
                  strategy=str(rng.choice(["keep_low", "keep_high"])))
    elif method == "streaming_llm":
        kw = dict(start_size=int(rng.integers(0, 9)), recent_size=int(rng.integers(0, 300)))
    elif method == "recent_only":
        kw = dict(window_size=cap)
    elif method == "h2o_l2":
        kw = dict(start_size=int(rng.integers(0, 9)), heavy_hitter_size=int(rng.integers(0, 100)),
                  recent_size=int(rng.integers(1, 300)))
    elif method == "snapkv_lite":
        kw = dict(observation_window=int(rng.integers(1, 64)), keep_size=cap, pooling_kernel=int(rng.integers(1, 10)))
    elif method == "pyramid_kv":
        kw = dict(base_size=cap, layer_decay=float(rng.choice([0.9, 0.8, 0.5, 1.0])), min_size=int(rng.integers(1, 100)),
                  profile=str(rng.choice(["exponential", "linear", "constant"])))
    else:
        soft = int(rng.integers(1, 300))
        hard = soft + int(rng.integers(1, 400))
        kw = dict(target_size=int(rng.integers(1, 400)), soft_limit=soft, hard_limit=hard,
                  keep_ratio_min=float(rng.choice([0.3, 0.1, 0.5])), keep_ratio_max=float(rng.choice([0.9, 0.7, 1.0])))
    kw["skip_layers"] = skip
    dtype = str(rng.choice(["f32", "f32", "bf16"]))
    style = str(rng.choice(["spread", "randn", "ties"]))
    return method, kw, seq_lens, int(rng.integers(1, 3)), int(rng.integers(1, 4)), int(rng.choice([8, 16])), dtype, style


@pytest.mark.parametrize("seed", range(48))
def test_random_calls_match_the_live_reference(ref, seed):
    rng = np.random.default_rng(9000 + seed)
    for _ in range(4):
        method, kw, seq_lens, B, H, D, dtype, style = draw_call(rng)
        layers = cases.make_cache(int(rng.integers(0, 1 << 30)), seq_lens, B, H, D, dtype, style)
        kv = []
        for K, _V in layers:
            k = to_torch(K, dtype)
            # V carries every row's own position, so the kept rows can be read back exactly (the reference never looks
            # at V when it selects)
            pos = torch.arange(k.size(2), dtype=torch.float32).view(1, 1, -1, 1).expand(k.shape).contiguous()
            kv.append((k, pos))
        what = (seed, method, kw, seq_lens, B, H, D, dtype, style)
        out = ref.get_compress_fn(method)(kv, **kw)
        res = O.METHODS[method](layers, dtype, **kw)
        plans = plan_for(method, seq_lens, kw)
        assert len(out) == len(kv) == len(res) == len(plans), what
        assert [int(k_out.size(2)) for k_out, _ in out] == O.out_lengths(layers, res) == [p.out_len for p in plans], what
        for li, ((k_in, v_in), (k_out, v_out)) in enumerate(zip(kv, out)):
            same = k_out is k_in and v_out is v_in
            assert same == res[li].untouched, (what, li)
            if same:
                continue
            assert bool(k_out._is_view()) == bool(res[li].is_view), (what, li)
            rows = v_out[..., 0].to(torch.int64).numpy()
            info = O.check_layer(layers[li][0], dtype, res[li], rows)
            assert info["valid"], (what, li, info)
            if dtype == "f32" and style != "ties":
                assert info["identical_heads"] == info["heads"], (what, li, info)
