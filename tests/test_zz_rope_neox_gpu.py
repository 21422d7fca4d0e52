"""GPU parity of `rotary_embedding_neox` (in-place NeoX RoPE from a cos|sin table; the HF-attention branch of tinychat,
tinychat/modules/fused_attn.py:61-79) through the C ABI and the `awq_inference_engine` plugin, against
oracle/layer_oracle.py and the stored output of the reference's own kernel rebuilt for sm_100a (tests/golden).

Tolerances: the kernel rounds ONCE to the element type from fp32 products, so against the float64 oracle an element
is equal or one ulp off; the reference's kernel multiplies and adds in the element type (up to three roundings per
output): <= 2 ulp of the larger operand, checked normwise per head.

The kernel's body is also checked without a GPU (tests/test_rope_neox_host.py).  This file sorts last on purpose: it
is the newest entry of the plugin."""
import ctypes
import os

import numpy as np
import pytest
import torch

import llm_awq_b200 as P
from oracle import layer_oracle as LO

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.float16, torch.bfloat16]
ULP = {torch.float16: 2.0 ** -10, torch.bfloat16: 2.0 ** -7}


def _inputs(tokens, qh, kh, hs, rot, dtype, seed, maxpos=211):
    g = torch.Generator().manual_seed(seed)
    name = "f16" if dtype == torch.float16 else "bf16"
    cache = torch.from_numpy(LO.neox_cos_sin_cache(rot, maxpos, 10000.0, name)).to(dtype)
    pos = torch.randint(0, maxpos, (tokens,), generator=g)
    q = torch.randn(tokens, qh, hs, generator=g).to(dtype)
    k = torch.randn(tokens, kh, hs, generator=g).to(dtype)
    return pos, q, k, cache


def _want(pos, q, k, hs, cache):
    return LO.rotary_embedding_neox(pos.numpy(), q.double().numpy(), k.double().numpy(), hs, cache.double().numpy(), "f64")


def _close(got, want64, dtype):
    g = got.double().cpu().numpy()
    return bool(np.all(np.abs(g - want64) <= ULP[dtype] * np.maximum(np.abs(want64), 2.0 ** -14)))


def _abi(pos, q, k, cache, hs, q_stride=None, k_stride=None):
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = P.lib().b200awq_rotary_embedding_neox(p(pos), p(q), p(k) if k.numel() else None, p(cache), q.shape[0], q.shape[1], k.shape[1], hs,
                                               cache.shape[1], q_stride or q.stride(0), k_stride or (k.stride(0) if k.numel() else 0),
                                               0 if q.dtype == torch.float16 else 1,
                                               ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    return rc


CASES = [  # tokens, q_heads, k_heads, head_size, rot_dim
    (1, 32, 32, 128, 128), (7, 32, 8, 128, 128), (2048, 32, 32, 128, 128), (5, 4, 4, 16, 16), (3, 8, 2, 64, 64),
    (2, 3, 1, 24, 16), (4, 2, 2, 12, 6), (6, 5, 5, 40, 40), (300, 40, 40, 128, 64), (1, 1, 1, 8, 8),
]


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("case", CASES)
def test_c_abi_vs_oracle(case, dtype):
    tokens, qh, kh, hs, rot = case
    pos, q, k, cache = _inputs(tokens, qh, kh, hs, rot, dtype, seed=tokens * 7 + hs)
    want_q, want_k = _want(pos, q, k, hs, cache)
    dq, dk, dpos, dcache = q.to(DEV), k.to(DEV), pos.to(DEV), cache.to(DEV)
    assert _abi(dpos, dq, dk, dcache, hs) == 0
    torch.cuda.synchronize()
    assert _close(dq, want_q, dtype) and _close(dk, want_k, dtype)
    assert torch.equal(dq[..., rot:].cpu(), q[..., rot:])                  # beyond rot_dim: untouched


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_plugin_signature_in_place_and_reference_shapes(dtype):
    """The call tinychat makes (fused_attn.py:61-79): positions [b, tokens], query / key [b, tokens, 1, heads, head_size]
    contiguous; in place, returns None."""
    eng = P.engine()
    b, t, H, D = 2, 9, 32, 128
    pos, q, k, cache = _inputs(b * t, H, H, D, D, dtype, seed=11)
    want_q, want_k = _want(pos, q, k, D, cache)
    dq, dk = q.view(b, t, 1, H, D).to(DEV), k.view(b, t, 1, H, D).to(DEV)
    ret = eng.rotary_embedding_neox(pos.view(b, t).to(DEV), dq, dk, D, cache.to(DEV))
    torch.cuda.synchronize()
    assert ret is None
    assert _close(dq.view(b * t, H, D), want_q, dtype) and _close(dk.view(b * t, H, D), want_k, dtype)


def test_plugin_rejects_what_it_cannot_take():
    eng = P.engine()
    pos, q, k, cache = _inputs(4, 2, 2, 16, 16, torch.float16, seed=1)
    dq, dk, dpos, dcache = (t.to(DEV) for t in (q.view(1, 4, 2, 16), k.view(1, 4, 2, 16), pos, cache))
    with pytest.raises(RuntimeError):
        eng.rotary_embedding_neox(dpos.int(), dq, dk, 16, dcache)          # positions must be int64
    with pytest.raises(RuntimeError):
        eng.rotary_embedding_neox(dpos, dq, dk, 16, dcache.float())        # table of another dtype
    with pytest.raises(RuntimeError):
        eng.rotary_embedding_neox(dpos, dq.float(), dk.float(), 16, dcache.float())   # fp32 is not dispatched
    with pytest.raises(RuntimeError):
        eng.rotary_embedding_neox(dpos, dq, dk, 8, dcache)                 # head_size does not match
    with pytest.raises(RuntimeError):
        eng.rotary_embedding_neox(dpos.cpu(), dq, dk, 16, dcache)          # host tensor
    # the C ABI's own checks
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    L = P.lib()
    q3, k3 = dq.view(4, 2, 16), dk.view(4, 2, 16)
    assert L.b200awq_rotary_embedding_neox(p(dpos), p(q3), p(k3), p(dcache), 4, 2, 2, 16, 15, 32, 32, 0, st) != 0   # odd rot_dim
    assert L.b200awq_rotary_embedding_neox(p(dpos), p(q3), p(k3), p(dcache), 4, 2, 2, 16, 32, 32, 32, 0, st) != 0   # rot_dim > head_size
    assert L.b200awq_rotary_embedding_neox(p(dpos), p(q3), p(k3), p(dcache), 4, 2, 2, 16, 16, 31, 32, 0, st) != 0   # stride < heads * head_size
    assert L.b200awq_rotary_embedding_neox(p(dpos), p(q3), p(k3), p(dcache), 4, 2, 2, 16, 16, 32, 32, 7, st) != 0   # dtype
    assert L.b200awq_rotary_embedding_neox(p(dpos), p(q3), p(k3), p(dcache), 0, 2, 2, 16, 16, 32, 32, 0, st) == 0   # no tokens: no-op
    torch.cuda.synchronize()
    assert torch.equal(q3.cpu(), q)                                       # nothing above touched the data


def test_views_into_a_fused_qkv_buffer_and_graph_replay():
    """query / key as strided views into a fused qkv output (C ABI: token strides), captured in a CUDA graph and
    replayed: each replay rotates once more (in place), the value heads are never touched."""
    tokens, qh, kh, hs = 6, 8, 2, 64
    row = (qh + 2 * kh) * hs
    g = torch.Generator().manual_seed(9)
    buf = torch.randn(tokens, row, generator=g).half()
    cache = torch.from_numpy(LO.neox_cos_sin_cache(hs, 50)).half()
    pos = torch.randint(0, 50, (tokens,), generator=g)
    q = buf[:, : qh * hs].view(tokens, qh, hs)
    k = buf[:, qh * hs: (qh + kh) * hs].view(tokens, kh, hs)
    w1q, w1k = _want(pos, q, k, hs, cache)
    rn = LO.O.rounder("f16")
    w2q, w2k = LO.rotary_embedding_neox(pos.numpy(), rn(w1q), rn(w1k), hs, cache.double().numpy(), "f64")
    dbuf, dpos, dcache = buf.to(DEV), pos.to(DEV), cache.to(DEV)
    dq = dbuf[:, : qh * hs].view(tokens, qh, hs)
    dk = dbuf[:, qh * hs: (qh + kh) * hs].view(tokens, kh, hs)
    scratch = dbuf.clone()                                                 # warm-up launch outside the capture
    assert _abi(dpos, scratch[:, : qh * hs].view(tokens, qh, hs), scratch[:, qh * hs: (qh + kh) * hs].view(tokens, kh, hs),
                dcache, hs, q_stride=row, k_stride=row) == 0
    torch.cuda.synchronize()
    gph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gph):
        assert _abi(dpos, dq, dk, dcache, hs, q_stride=row, k_stride=row) == 0
    gph.replay()
    torch.cuda.synchronize()
    assert _close(dq, w1q, torch.float16) and _close(dk, w1k, torch.float16)
    gph.replay()
    torch.cuda.synchronize()
    # the first rotation may sit one ulp from the oracle's rounding: compare the second per head, 3 ulp of its largest element
    for got, want in ((dq, w2q), (dk, w2k)):
        g64 = got.double().cpu().numpy()
        assert np.all(np.abs(g64 - want) <= 3 * ULP[torch.float16] * np.abs(want).max(axis=-1, keepdims=True))
    assert torch.equal(dbuf[:, (qh + kh) * hs:].cpu(), buf[:, (qh + kh) * hs:])


def rope_ref_inputs(dtype, device):
    """pos [1, 33], q and k [1, 33, 1, 32, 128] and the cos|sin table of test_vs_reference_kernel, on `device`; the
    reference kernel's in-place result on them is stored in tests/golden/reference_kernels.npz
    (tests/golden/make_golden.py --kernels)."""
    b, t, H, D = 1, 33, 32, 128
    pos, q, k, cache = _inputs(b * t, H, H, D, D, dtype, seed=21)
    return pos.view(b, t).to(device), q.view(b, t, 1, H, D).to(device), k.view(b, t, 1, H, D).to(device), cache.to(device)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_vs_reference_kernel(dtype):
    eng = P.engine()
    dpos, mine_q, mine_k, dcache = rope_ref_inputs(dtype, DEV)
    q, k = mine_q.cpu(), mine_k.cpu()
    eng.rotary_embedding_neox(dpos, mine_q, mine_k, mine_q.shape[-1], dcache)
    torch.cuda.synchronize()
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_kernels.npz"))
    tag = "f16" if dtype == torch.float16 else "bf16"
    for nm, a, x in (("q", mine_q, q), ("k", mine_k, k)):
        idx = torch.from_numpy(gold[f"rope_{tag}_{nm}_idx"]).long()
        D = x.shape[-1]
        r64 = torch.from_numpy(gold[f"rope_{tag}_{nm}"]).view(dtype).double()
        a64 = a.cpu().reshape(-1, D)[idx].double()
        scale = x.reshape(-1, D)[idx].double().abs().amax(dim=-1, keepdim=True)   # |x'| <= |x| + |y| <= 2 max|head|
        assert bool(((a64 - r64).abs() <= 4 * ULP[dtype] * scale).all())
        num, den = (a64 - r64).norm(dim=-1), r64.norm(dim=-1)
        assert bool((num <= 2 * ULP[dtype] * den).all())
