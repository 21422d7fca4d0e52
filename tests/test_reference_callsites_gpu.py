"""The reference's OWN call sites and what they compute, against this repo's modules on the GPU (SURVEY.md §8 a13, a3):

    awq.quantize.qmodule.WQLinear                  forward: qmodule.py:201-224 (GEMV for < 8 tokens, else GEMM, + bias)
    tinychat.modules.fused_mlp.QuantLlamaMLP       our_llama_mlp: fused_mlp.py:36-83 (both branches, incl. the GEMM
                                                   branch's `scaled_zeros - 8 * scales`)
    tinychat.modules.fused_attn.make_quant_attn    the fused-QKV WQLinear built by concatenating packed tensors,
                                                   fused_attn.py:566-594

tests/golden/reference_callsites.npz holds what those call sites, unmodified, returned when executed on CPU over
oracle-backed engine calls, and which engine entry each made (tests/golden/make_golden.py::callsites_golden), on the
inputs regenerated here from the same seeds.  The repo's drop-ins (llm_awq_b200.WQLinear, llm_awq_b200.fused_mlp.
QuantLlamaMLP with the reference's GEMM-branch zeros) must make the same entry calls on the plugin and return the same
results; every result is also checked against the CPU oracle."""
import os

import numpy as np
import pytest
import torch

import llm_awq_b200 as P
from llm_awq_b200.fused_mlp import QuantLlamaMLP
from oracle import layer_oracle as LO
from oracle import w4a16_oracle as O
from awq_testutil import dt_name, gen_layer, gen_x, np64, oracle_forward, rel_err
from test_gpu_parity import check

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
WQ_SHAPES = [(1, 1), (1, 7), (1, 8), (2, 40), (1, 300)]
MLP_TOKENS = [1, 4, 7, 8, 64, 300]
QKV_TOKENS = [1, 5, 16, 130]


def callsite_rows(M):
    """Rows of an [M, N] output kept in the golden file (at every other column): all of them up to 4, else 4 seeded
    ones."""
    return np.arange(M) if M <= 4 else np.sort(np.random.default_rng(M).choice(M, 4, replace=False))


def layer_bias(N, dtype, seed):
    g = torch.Generator().manual_seed(seed + 1)
    return (torch.randn(N, generator=g) * 0.1).to(dtype)


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_callsites.npz"))


def _wqlinear(K, N, dtype, seed, bias=False):
    """A WQLinear with synthetic packed buffers (the constructor zero-fills them, qmodule.py:98-137)."""
    m = P.WQLinear(4, 128, K, N, bias, DEV, dtype=dtype)
    qw, s, z = gen_layer(N, K, dtype, seed=seed, device=DEV)
    assert m.qweight.shape == qw.shape and m.scales.shape == s.shape and m.scaled_zeros.shape == z.shape
    m.qweight, m.scales, m.scaled_zeros = qw, s, z
    if bias:
        m.bias = layer_bias(N, dtype, seed).to(DEV)
    return m


def _entries(gold, key, tokens):
    """The reference made one engine call per linear, the GEMV entry below 8 tokens and the GEMM entry from 8."""
    calls = [str(c) for c in gold[key + "_calls"]]
    assert set(calls) == {"gemv" if tokens < 8 else "gemm"}
    return len(calls)


def _sample(y, M):
    return np64(y.reshape(M, -1))[callsite_rows(M)][:, ::2]


def _stored(gold, key, dtype):
    return np64(torch.from_numpy(gold[key]).view(dtype))


@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["f16", "bf16"])
@pytest.mark.parametrize("shape", WQ_SHAPES, ids=str)
@pytest.mark.parametrize("bias", [False, True])
def test_unmodified_reference_wqlinear_forward(gold, shape, dtype, bias):
    """llm_awq_b200.WQLinear.forward against what the reference's unmodified WQLinear.forward returned (stored): the same
    engine entry, one launch, the same output; the reference's code does not run here."""
    K, N = 1024, 768
    M = shape[0] * shape[1]
    key = f"wq_{dt_name(dtype)}_b{int(bias)}_{shape[0]}x{shape[1]}"
    m = _wqlinear(K, N, dtype, seed=5, bias=bias)
    x = gen_x(M, K, dtype, seed=shape[1], device=DEV).view(*shape, K)
    before = P.engine().launch_count()
    y = m(x)
    torch.cuda.synchronize()
    assert P.engine().launch_count() == before + _entries(gold, key, M) and y.shape == (*shape, N)
    want = oracle_forward(x.view(-1, K), m.qweight, m.scales, m.scaled_zeros, dtype)
    if bias:
        want = O.rounder(dt_name(dtype))(want) + np64(m.bias)   # the reference adds the bias to the ROUNDED output (:221)
    tol = 1e-3 if not bias else (1e-3 if dtype == torch.float16 else 6e-3)
    check(y.view(-1, N), want, dtype, tol=tol)
    assert rel_err(_sample(y, M), _stored(gold, key + "_y", dtype)) <= tol


@pytest.mark.parametrize("tokens", MLP_TOKENS)
def test_unmodified_reference_fused_mlp_both_branches(gold, tokens):
    """QuantLlamaMLP.our_llama_mlp: < 8 tokens -> two GEMV calls with the zeros as stored (fused_mlp.py:40-60);
    otherwise two GEMM calls with `scaled_zeros - 8 * scales` (:65-77; the tensor expression is evaluated in fp16 by
    torch before the call, and the oracle is given exactly that tensor: "use the zeros you are given").  The reference's
    code does not run here: its stored output is compared with the drop-in llm_awq_b200.fused_mlp.QuantLlamaMLP, which
    makes one engine call of the fused front half in place of the reference's two linears + F.silu + multiply.  That
    call launches the one-kernel gate+up+SiLU*mul for one token, else the reference's linears (one launch each) and one
    SiLU*mul kernel."""
    dtype, H, I = torch.float16, 1024, 2816
    gate, up, down = _wqlinear(H, I, dtype, 11), _wqlinear(H, I, dtype, 12), _wqlinear(I, H, dtype, 13)
    mlp = QuantLlamaMLP(gate, down, up, legacy_gemm_zero_offset=True)
    ref_calls = _entries(gold, f"mlp_t{tokens}", tokens)
    assert ref_calls == 2                                        # gate_proj and up_proj
    x = (gen_x(tokens, H, dtype, seed=tokens, device=DEV) * 0.5).view(1, tokens, H)
    before = P.engine().launch_count()
    c = mlp.our_llama_mlp(x)
    torch.cuda.synchronize()
    assert P.engine().launch_count() - before == (1 if tokens == 1 else ref_calls + 1)
    assert c.shape == (1, tokens, I)
    if tokens < 8:
        gz, uz = gate.scaled_zeros, up.scaled_zeros
    else:
        gz, uz = gate.scaled_zeros - 8 * gate.scales, up.scaled_zeros - 8 * up.scales
    want = LO.mlp_front(np64(x.view(tokens, H)), (gate.qweight.cpu().numpy(), np64(gate.scales), np64(gz)),
                        (up.qweight.cpu().numpy(), np64(up.scales), np64(uz)), dtype="f16")
    # products of two rounded factors: 2 ulp of fp16 normwise
    assert rel_err(np64(c.view(tokens, I)), want) < 1.5e-3
    assert rel_err(_sample(c, tokens), _stored(gold, f"mlp_t{tokens}_c", dtype)) < 1.5e-3
    y = mlp(x)                                                   # + down_proj through WQLinear.forward
    torch.cuda.synchronize()
    want_y = oracle_forward(c.view(tokens, I), down.qweight, down.scales, down.scaled_zeros, dtype)
    check(y.view(tokens, H), want_y, dtype)


def test_unmodified_reference_make_quant_attn_concatenation(gold):
    """make_quant_attn (fused_attn.py:556-640) builds the fused QKV layer by torch.cat of qweight (dim 0) / scales /
    scaled_zeros (dim 1): the same concatenation here must give the buffers the reference built (stored shapes and
    sums), and [q; k; v] of the three separate projections through the plugin, as the reference's fused layer returned
    them, for decode and prefill token counts.  The reference's code does not run here."""
    dtype, H, KV = torch.float16, 1024, 256
    parts = [_wqlinear(H, H, dtype, 21), _wqlinear(H, KV, dtype, 22), _wqlinear(H, KV, dtype, 23)]
    qkv = P.WQLinear(4, 128, H, H + 2 * KV, False, DEV, dtype=dtype)
    qkv.qweight = torch.cat([p.qweight for p in parts], dim=0)
    qkv.scales = torch.cat([p.scales for p in parts], dim=1).contiguous()
    qkv.scaled_zeros = torch.cat([p.scaled_zeros for p in parts], dim=1).contiguous()
    for nm in ("qweight", "scales", "scaled_zeros"):
        t = getattr(qkv, nm).cpu()
        assert tuple(t.shape) == tuple(gold[f"qkv_{nm}_shape"])
        s = t.float().numpy().astype(np.float64).sum() if t.is_floating_point() else t.numpy().astype(np.int64).sum()
        assert s == gold[f"qkv_{nm}_sum"], nm
    for tokens in QKV_TOKENS:
        key = f"qkv_t{tokens}"
        x = gen_x(tokens, H, dtype, seed=30 + tokens, device=DEV).view(1, tokens, H)
        before = P.engine().launch_count()
        y = qkv(x)
        torch.cuda.synchronize()
        assert P.engine().launch_count() == before + _entries(gold, key, tokens)
        want = np.concatenate([oracle_forward(x.view(tokens, H), p.qweight, p.scales, p.scaled_zeros, dtype) for p in parts], axis=1)
        check(y.view(tokens, -1), want, dtype)
        assert rel_err(_sample(y, tokens), _stored(gold, key + "_y", dtype)) <= 1e-3
