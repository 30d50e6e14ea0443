"""No GPU: kvc_query_window_push's exported symbol and refusals (each status returned before any CUDA call: on a machine
without a device a CUDA call would answer KVC_ERR_CUDA), and every ValueError of SnapKVQueryWindow, of the methods that
take it, and of the harnesses' scores="queries" checks, which run before the first forward."""

import ctypes as C
from types import SimpleNamespace

import pytest
import torch

import kvcompress
from kvcompress import QueryCapture, SnapKVQueryWindow, _engine
from kvcompress.benchmark import measure_generation_metrics
from kvcompress.evaluate import evaluate_with_compression

BF16, F16, F32 = 2, 1, 0


@pytest.fixture(scope="module")
def lib():
    return _engine.load_library()


def test_symbol_is_exported(lib):
    assert hasattr(lib, "kvc_query_window_push")
    assert _engine._QWIN.size == 64


def push(lib, shape, window, recs, n=None):
    buf = b"".join(_engine._QWIN.pack(*r) for r in recs)
    return lib.kvc_query_window_push(shape, window, len(recs) if n is None else n, buf if recs else None, None)


def rec(q=0x1000, qs=(8192, 1024, 128), w=0x2000, ws=(4096, 512), filled=0, n_new=1):
    return (q, qs[0], qs[1], qs[2], w, ws[0], ws[1], filled, n_new)


@pytest.mark.parametrize("why,shape,window,recs,status", [
    ("no shape", None, 8, [rec()], 1),
    ("batch 0", (0, 4, 64, BF16, 0), 8, [rec()], 1),
    ("window 0", (1, 4, 64, BF16, 0), 0, [rec()], 1),
    ("window 129", (1, 4, 64, BF16, 0), 129, [rec()], 1),
    ("fp32", (1, 4, 64, F32, 0), 8, [rec()], 2),
    ("NULL q_new", (1, 4, 64, BF16, 0), 8, [rec(q=0)], 1),
    ("NULL window", (1, 4, 64, BF16, 0), 8, [rec(w=0)], 1),
    ("filled < 0", (1, 4, 64, BF16, 0), 8, [rec(filled=-1)], 1),
    ("filled > W", (1, 4, 64, BF16, 0), 8, [rec(filled=9)], 1),
    ("n_new < 0", (1, 4, 64, BF16, 0), 8, [rec(n_new=-1)], 1),
    ("row width 8 bytes", (1, 4, 4, F16, 0), 8, [rec()], 2),
    ("q base", (1, 4, 64, BF16, 0), 8, [rec(q=0x1008)], 2),
    ("window base", (1, 4, 64, BF16, 0), 8, [rec(w=0x2002)], 2),
    ("q stride s", (1, 4, 64, F16, 0), 8, [rec(qs=(8192, 1024, 68))], 2),
    ("q stride h", (1, 4, 64, BF16, 0), 8, [rec(qs=(8192, 1028, 128))], 2),
    ("window stride b", (1, 4, 64, BF16, 0), 8, [rec(ws=(4100, 512))], 2),
    ("second layer", (1, 4, 64, BF16, 0), 8, [rec(), rec(filled=12)], 1),
])
def test_refusals_before_any_cuda_call(lib, why, shape, window, recs, status):
    packed = None if shape is None else _engine._SHAPE.pack(*shape)
    assert push(lib, packed, window, recs) == status, why


def test_null_records_and_empty_calls(lib):
    shape = _engine._SHAPE.pack(1, 4, 64, BF16, 0)
    assert lib.kvc_query_window_push(shape, 8, 1, None, None) == 1
    assert lib.kvc_query_window_push(shape, 8, -1, None, None) == 1
    assert lib.kvc_query_window_push(shape, 8, 0, None, None) == 0


def cpu_window(L=2, B=1, Hq=4, D=64, W=8):
    return SnapKVQueryWindow(L, B, Hq, D, W, torch.bfloat16, device="cpu")


def fake_capture(L, queries, scaling=None, masks=None):
    cap = QueryCapture(L)
    for l, q in enumerate(queries):
        cap._record(l, q, None, None if masks is None else masks[l],
                    q.size(-1) ** -0.5 if scaling is None else scaling)
    return cap


def test_constructor_refusals():
    with pytest.raises(ValueError, match="window"):
        SnapKVQueryWindow(2, 1, 4, 64, 0, torch.bfloat16, device="cpu")
    with pytest.raises(ValueError, match="window"):
        SnapKVQueryWindow(2, 1, 4, 64, 129, torch.bfloat16, device="cpu")
    with pytest.raises(ValueError, match="bfloat16/float16"):
        SnapKVQueryWindow(2, 1, 4, 64, 8, torch.float32, device="cpu")
    w = cpu_window()
    assert [tuple(q.shape) for q in w.queries] == [(1, 4, 8, 64)] * 2 and w.filled == [0, 0]


def test_push_refuses_other_scalings_and_masks():
    w = cpu_window()
    q = [torch.zeros(1, 4, 1, 64, dtype=torch.bfloat16) for _ in range(2)]
    with pytest.raises(ValueError, match="scaling"):
        w.push(fake_capture(2, q, scaling=0.1))
    mask = torch.ones(1, 1, 1, 9, dtype=torch.bool)
    with pytest.raises(ValueError, match="mask"):
        w.push(fake_capture(2, q, masks=[None, mask]))
    with pytest.raises(ValueError, match="layers"):
        w.push(q[:1])
    assert w.filled == [0, 0]  # nothing was pushed


def test_compression_refuses_a_short_or_mismatched_window():
    L, S, W = 2, 100, 8
    kv = [(torch.zeros(1, 4, S, 64, dtype=torch.bfloat16), torch.zeros(1, 4, S, 64, dtype=torch.bfloat16))
          for _ in range(L)]
    w = cpu_window(L=L, W=W)
    w.filled = [W, W - 1]
    with pytest.raises(ValueError, match=r"layers \[1\]"):
        kvcompress.snapkv_lite_compress(kv, observation_window=W, keep_size=32, obs_queries=w)
    w.filled = [W, W]
    with pytest.raises(ValueError, match="observation_window"):
        kvcompress.snapkv_lite_compress(kv, observation_window=16, keep_size=32, obs_queries=w)
    w.reset()
    assert w.filled == [0, 0]
    # a layer that does not vote (skipped) may be short
    w.filled = [W, 0]
    assert w.queries_for(W, [0]) is w.queries


class FakeModel(torch.nn.Module):
    """Config and parameters of a model; any forward is a test failure."""

    def __init__(self, dtype=torch.bfloat16, heads=8, kv_heads=2, head_dim=64):
        super().__init__()
        self.config = SimpleNamespace(num_hidden_layers=2, num_attention_heads=heads, num_key_value_heads=kv_heads,
                                      hidden_size=heads * head_dim, head_dim=head_dim, vocab_size=16)
        self.w = torch.nn.Parameter(torch.zeros(1, dtype=dtype))

    def forward(self, *args, **kwargs):
        raise AssertionError("a forward ran before the argument checks")


@pytest.mark.parametrize("harness", ["evaluate", "generate"])
@pytest.mark.parametrize("model,compress_fn,kwargs,match", [
    (FakeModel(), kvcompress.h2o_l2_compress, {}, "snapkv_lite_compress"),
    (FakeModel(dtype=torch.float32), kvcompress.snapkv_lite_compress, {}, "bfloat16/float16"),
    (FakeModel(heads=16, kv_heads=2), kvcompress.snapkv_lite_compress, {"observation_window": 32}, "128 query rows"),
    (FakeModel(heads=8, kv_heads=2, head_dim=96), kvcompress.snapkv_lite_compress, {}, "head_dim"),
])
def test_harness_checks_run_before_the_first_forward(harness, model, compress_fn, kwargs, match):
    ids = torch.zeros(1, 40, dtype=torch.long)
    fn = evaluate_with_compression if harness == "evaluate" else measure_generation_metrics
    with pytest.raises(ValueError, match=match):
        fn(model, input_ids=ids, compress_fn=compress_fn, compress_kwargs=kwargs, scores="queries")


@pytest.mark.parametrize("fn", [evaluate_with_compression, measure_generation_metrics])
def test_unknown_score_source(fn):
    with pytest.raises(ValueError, match="scores"):
        fn(FakeModel(), input_ids=torch.zeros(1, 40, dtype=torch.long), compress_fn=kvcompress.snapkv_lite_compress,
           scores="attentions")
