"""GPU parity of `single_query_attention` for any query-to-KV head ratio G = heads / kv_heads and every head dimension
the reference's FasterTransformer kernel accepts: the CUDA-core kernel for G <= 8 (any head_dim that is a multiple of
8 up to 256) and the tensor-core kernel for 9 <= G <= 128 (head_dim a multiple of 16 up to 256), against
oracle/layer_oracle.py (head h reads KV head h // G, the reference's hi / kv_rep) and torch SDPA.

Tolerances as in tests/test_attention_gpu.py: 2e-3 normwise for fp16, 8e-3 for bf16.  The tensor-core kernel rounds
the probabilities to the element type before the product with V, as the reference does."""
import ctypes

import numpy as np
import pytest
import torch

import llm_awq_b200 as P
from oracle import layer_oracle as LO
from awq_testutil import dt_name, np64, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ERR_SHAPE, ERR_WORKSPACE = -1, -6


def _tol(dtype):
    return 2e-3 if dtype == torch.float16 else 8e-3


def _caches(B, Hkv, D, L, dtype, fill_to, seed):
    g = torch.Generator().manual_seed(seed)
    kc = torch.zeros(B, Hkv, D // 8, L, 8)
    vc = torch.zeros(B, Hkv, L, D)
    kc[:, :, :, :fill_to] = torch.randn(B, Hkv, D // 8, fill_to, 8, generator=g)
    vc[:, :, :fill_to] = torch.randn(B, Hkv, fill_to, D, generator=g)
    return kc.to(dtype).to(DEV), vc.to(dtype).to(DEV)


def _fused_qkv(B, H, Hkv, D, dtype, seed):
    """q, k, v as views into one fused QKV output (batch stride (H + 2 Hkv) * D > H * D), as tinychat views them."""
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B, 1, H + 2 * Hkv, D, generator=g).to(dtype).to(DEV)
    return qkv[:, 0, :H], qkv[:, 0, H:H + Hkv], qkv[:, 0, H + Hkv:]


def _check_against_oracle(B, H, Hkv, D, L, t, dtype, seed):
    eng = P.engine()
    q, k, v = _fused_qkv(B, H, Hkv, D, dtype, seed)
    kc, vc = _caches(B, Hkv, D, L, dtype, min(t, L), seed=seed + 1)
    kc64, vc64 = np64(kc), np64(vc)
    out = eng.single_query_attention(q, k, v, kc, vc, None, None, t, D, 1000000.0, 1.0, True)
    torch.cuda.synchronize()
    want = LO.single_query_attention(np64(q), np64(k), np64(v), kc64, vc64, t, D, 1000000.0, 1.0, True, dt_name(dtype))
    assert out.shape == (B, H, D)
    assert rel_err(np64(out), want) < _tol(dtype)
    # the cache update: v of this step bit for bit, the rotated k to fp32-angle accuracy, every other slot untouched
    assert np.array_equal(np64(vc), vc64)
    slot = t % L
    got_kc = np64(kc)
    assert np.abs(got_kc[:, :, :, slot] - kc64[:, :, :, slot]).max() <= 2e-3 * np.abs(kc64[:, :, :, slot]).max()
    mask = np.ones(L, dtype=bool)
    mask[slot] = False
    assert np.array_equal(got_kc[:, :, :, mask], kc64[:, :, :, mask])


# (heads, kv_heads, head_dim): Llama-3.2-3B, Qwen2.5-14B, Qwen2-1.5B, Qwen2-7B, Qwen2-0.5B, Falcon-40B, Falcon-7B-style
# multi-query, multi-query at d 128 and d 256
RATIOS = [(24, 8, 128), (40, 8, 128), (12, 2, 128), (28, 4, 128), (14, 2, 64), (128, 8, 64), (71, 1, 64), (128, 1, 128),
          (32, 1, 256)]
# (max_len, timestep): empty cache, one CTA, split over CTAs, a full cache, a wrapped cache (t >= L)
CONTEXTS = {"t0": (256, 0), "short": (256, 37), "long": (2048, 1500), "full": (512, 511), "wrapped": (512, 700)}


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("ctx", list(CONTEXTS))
@pytest.mark.parametrize("H,Hkv,D", RATIOS, ids=["%d-%d-d%d" % r for r in RATIOS])
def test_ratio_head_dim_grid_vs_oracle(H, Hkv, D, ctx, dtype):
    L, t = CONTEXTS[ctx]
    _check_against_oracle(2, H, Hkv, D, L, t, dtype, seed=H * 7 + D + t)


SMALL_DIMS = [(G, D) for D in (48, 80, 96, 112, 160) for G in (1, 7)] + [(16, 80)]


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("G,D", SMALL_DIMS, ids=["G%d-d%d" % s for s in SMALL_DIMS])
def test_head_dims_not_dividing_2048(G, D, dtype):
    """Head dims of the reference's set that 2048 is not a multiple of (plus 96 and 160): on the CUDA-core kernel the
    P.V loop leaves 256 % (D / 8) threads idle; one tensor-core case at d 80 (a d % 32 == 16 tail)."""
    Hkv = 2
    _check_against_oracle(2, G * Hkv, Hkv, D, 1024, 700, dtype, seed=G * 100 + D)


def test_length_per_sample_partial_interleaved_rope_tensor_cores():
    eng = P.engine()
    dtype, B, H, Hkv, D, L = torch.float16, 2, 32, 2, 128, 1024
    g = torch.Generator().manual_seed(11)
    q = torch.randn(B, H, D, generator=g).to(dtype).to(DEV)
    k = torch.randn(B, Hkv, D, generator=g).to(dtype).to(DEV)
    v = torch.randn(B, Hkv, D, generator=g).to(dtype).to(DEV)
    kc, vc = _caches(B, Hkv, D, L, dtype, L, seed=12)
    kc64, vc64 = np64(kc), np64(vc)
    lps = torch.tensor([5, 900], dtype=torch.int32, device=DEV)
    out = eng.single_query_attention(q, k, v, kc, vc, lps, None, 950, 64, 10000.0, 0.5, False)   # partial, interleaved
    torch.cuda.synchronize()
    want = LO.single_query_attention(np64(q), np64(k), np64(v), kc64, vc64, 950, 64, 10000.0, 0.5, False, "f16",
                                     length_per_sample=[5, 900])
    assert rel_err(np64(out), want) < 2e-3 and rel_err(np64(kc), kc64) < 1e-3
    assert np.array_equal(np64(vc), vc64)


@pytest.mark.parametrize("H,Hkv,D", [(28, 4, 128), (71, 1, 64)], ids=["G7", "G71"])
def test_decode_loop_matches_sdpa(H, Hkv, D):
    """40 decode steps from an empty cache against torch SDPA on the keys read back from the cache layout: the cache
    writes of each step feed the later steps."""
    eng = P.engine()
    dtype, B, L = torch.float16, 1, 64
    kc = torch.zeros(B, Hkv, D // 8, L, 8, dtype=dtype, device=DEV)
    vc = torch.zeros(B, Hkv, L, D, dtype=dtype, device=DEV)
    g = torch.Generator().manual_seed(H)
    for t in range(40):
        qkv = torch.randn(B, 1, H + 2 * Hkv, D, generator=g).to(dtype).to(DEV)
        q, k, v = qkv[:, 0, :H], qkv[:, 0, H:H + Hkv], qkv[:, 0, H + Hkv:]
        out = eng.single_query_attention(q, k, v, kc, vc, None, None, t, D, 10000.0, 1.0, True)
        keys = kc[:, :, :, :t + 1].permute(0, 1, 3, 2, 4).reshape(B, Hkv, t + 1, D).float()
        vals = vc[:, :, :t + 1].float()
        qr = torch.from_numpy(LO.rope_rotate(np64(q), t, D, 10000.0, 1.0, True, "f16")).float().to(DEV)
        ref = torch.nn.functional.scaled_dot_product_attention(qr.view(B, H, 1, D), keys.repeat_interleave(H // Hkv, 1),
                                                               vals.repeat_interleave(H // Hkv, 1))
        assert rel_err(np64(out), np64(ref.view(B, H, D))) < 2e-3, t


def _abi(lib, q, k, v, kc, vc, out, H, Hkv, D, L, t, ws, ws_bytes, stream):
    p = lambda x: ctypes.c_void_p(x.data_ptr())
    B = q.shape[0]
    return lib.b200awq_single_query_attention(p(q), p(k), p(v), p(kc), p(vc), p(out), None, B, H, Hkv, D, L, t,
                                              q.stride(0), k.stride(0), v.stride(0), D, 10000.0, 1.0, 1,
                                              0 if q.dtype == torch.float16 else 1, p(ws), ws_bytes,
                                              ctypes.c_void_p(stream))


def test_graph_replay_split_context_leaves_counters_zero():
    """G = 16, context 4096 split over CTAs, captured on a side stream: replays agree bit for bit with the eager call and
    the arrival counters at the start of the workspace are back at zero."""
    eng, lib = P.engine(), P.lib()
    dtype, B, H, Hkv, D, L, t = torch.float16, 1, 128, 8, 64, 4096, 4095
    q, k, v = _fused_qkv(B, H, Hkv, D, dtype, seed=21)
    kc, vc = _caches(B, Hkv, D, L, dtype, t, seed=22)
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        first = eng.single_query_attention(q, k, v, kc, vc, None, None, t, D, 10000.0, 1.0, True).clone()
        gr = torch.cuda.CUDAGraph()
        side.synchronize()
        with torch.cuda.graph(gr, stream=side):
            o = eng.single_query_attention(q, k, v, kc, vc, None, None, t, D, 10000.0, 1.0, True)
        for _ in range(3):
            gr.replay()
            side.synchronize()
            assert torch.equal(o, first)
    want = LO.single_query_attention(np64(q), np64(k), np64(v), np64(kc), np64(vc), t, D, 10000.0, 1.0, True, "f16")
    assert rel_err(np64(first), want) < 2e-3
    # the same launch through the C ABI on a workspace of our own: counters zero after eager calls and graph replays
    need = lib.b200awq_single_query_attention_workspace_bytes(B, H, Hkv, D, L)
    ws = torch.zeros(need, dtype=torch.uint8, device=DEV)
    out = torch.empty(B, H, D, dtype=dtype, device=DEV)
    with torch.cuda.stream(side):
        assert _abi(lib, q, k, v, kc, vc, out, H, Hkv, D, L, t, ws, need, side.cuda_stream) == 0
        gr2 = torch.cuda.CUDAGraph()
        side.synchronize()
        with torch.cuda.graph(gr2, stream=side):
            _abi(lib, q, k, v, kc, vc, out, H, Hkv, D, L, t, ws, need, side.cuda_stream)
        for _ in range(3):
            gr2.replay()
        side.synchronize()
    assert torch.equal(out, first)
    assert int(ws[:4096 * 4].count_nonzero()) == 0


def test_c_abi_group_and_head_dim_limits():
    lib = P.lib()
    dtype, B, D, L, t = torch.float16, 1, 64, 128, 100
    st = torch.cuda.current_stream().cuda_stream

    def call(H, Hkv, D, short=0):
        q = torch.randn(B, H, D, device=DEV).to(dtype)
        k = torch.randn(B, Hkv, D, device=DEV).to(dtype)
        v = torch.randn(B, Hkv, D, device=DEV).to(dtype)
        kc, vc = _caches(B, Hkv, D, L, dtype, t, seed=H)
        out = torch.empty(B, H, D, dtype=dtype, device=DEV)
        need = lib.b200awq_single_query_attention_workspace_bytes(B, H, Hkv, D, L)
        ws = torch.zeros(max(need, 16), dtype=torch.uint8, device=DEV)
        want = LO.single_query_attention(np64(q), np64(k), np64(v), np64(kc), np64(vc), t, D, 10000.0, 1.0, True, "f16")
        rc = _abi(lib, q, k, v, kc, vc, out, H, Hkv, D, L, t, ws, need - short, st)
        torch.cuda.synchronize()
        return rc, out, want

    rc, out, want = call(128, 1, 64)                                   # G = 128: the widest group served
    assert rc == 0 and rel_err(np64(out), want) < 2e-3
    assert call(129, 1, 64)[0] == ERR_SHAPE                            # G = 129
    assert call(16, 1, 40)[0] == ERR_SHAPE                             # head_dim 40 on the tensor-core kernel
    assert call(16, 1, 64, short=1)[0] == ERR_WORKSPACE                # workspace one byte short
    assert call(7, 1, 64, short=1)[0] == ERR_WORKSPACE
    rc, out, want = call(4, 1, 40)                                     # head_dim 40 is fine for G <= 8
    assert rc == 0 and rel_err(np64(out), want) < 2e-3
