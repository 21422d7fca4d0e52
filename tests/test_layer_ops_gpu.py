"""GPU parity of the ops adjacent to the W4A16 linears (SURVEY.md §8f): RMSNorm (`layernorm_forward_cuda`) and the
fused gate+up+SiLU*mul front half of the MLP, through the C ABI and the `awq_inference_engine` plugin, against
oracle/layer_oracle.py and the stored output of the reference's own kernel rebuilt for sm_100a (tests/golden).

Tolerances: both ops round ONCE to the element type from fp32, so against the float64 oracle rounded to the type
an element is either equal or one ulp off (fp32 vs fp64 statistics flip a few roundings); the tests bound the
fraction of one-ulp elements and the normwise error (1e-3, north_star)."""
import ctypes
import os

import numpy as np
import pytest
import torch

import llm_awq_b200 as P
from oracle import layer_oracle as LO
from oracle import w4a16_oracle as O
from awq_testutil import dt_name, gen_layer, gen_x, np64, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DTYPES = [torch.float16, torch.bfloat16]


def _ulps(y, want, dtype):
    """|y - want| in units of the element type's spacing at `want`."""
    yi = y.view(torch.int16).to(torch.int32)
    wi = want.view(torch.int16).to(torch.int32)
    return (yi - wi).abs()   # same sign and finite: adjacent bit patterns are adjacent values


def rmsnorm_ref_inputs(dtype, device):
    """x [2, 33, 4096] and gamma of test_rmsnorm_plugin_signature_and_reference_kernel; the reference kernel's output on
    them is stored in tests/golden/reference_kernels.npz (tests/golden/make_golden.py --kernels)."""
    x = (gen_x(2 * 33, 4096, dtype, seed=5, device=device) * 2.0).view(2, 33, 4096)
    gamma = (1.0 + 0.1 * gen_x(1, 4096, dtype, seed=6, device=device)).view(4096)
    return x, gamma


def _rmsnorm_abi(x, g, eps):
    y = torch.empty_like(x)
    m, n = x.numel() // x.shape[-1], x.shape[-1]
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = P.lib().b200awq_rmsnorm(p(x), p(g), p(y), m, n, eps, 0 if x.dtype == torch.float16 else 1,
                                 ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, P.lib().b200awq_strerror(rc)
    return y


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("m,n", [(1, 4096), (7, 4096), (2048, 4096), (3, 8192), (64, 14336), (5, 128), (2, 8),
                                 (9, 5120), (4, 11008), (3, 100), (2, 4100), (1, 32768), (2, 40000)])
def test_rmsnorm_vs_oracle(m, n, dtype):
    g = torch.Generator().manual_seed(m * 131 + n)
    x = (torch.randn(m, n, generator=g) * 1.7).to(dtype).to(DEV)
    gamma = (1.0 + 0.2 * torch.randn(n, generator=g)).to(dtype).to(DEV)
    eps = 1e-5
    y = _rmsnorm_abi(x, gamma, eps)
    torch.cuda.synchronize()
    want64 = LO.rmsnorm(np64(x), np64(gamma), eps, dt_name(dtype))
    want = torch.from_numpy(want64).to(dtype).to(DEV)
    u = _ulps(y, want, dtype)
    assert int(u.max()) <= 1
    assert float((u > 0).float().mean()) < 2e-3       # fp32 vs float64 statistics: a few roundings flip
    # against the UNROUNDED result the error is the output rounding itself: 2^-12 / sqrt(3) normwise for fp16,
    # 2^-9 / sqrt(3) = 1.1e-3 .. 1.8e-3 for bf16 (the 1e-3 of north_star is an fp16 figure; see BASELINE.md)
    tol = 1e-3 if dtype == torch.float16 else 4e-3
    assert rel_err(np64(y), LO.rmsnorm(np64(x), np64(gamma), eps, dt_name(dtype), rounded=False)) < tol


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_rmsnorm_plugin_signature_and_reference_kernel(dtype):
    """layernorm_forward_cuda(input [b, s, c], gamma, out, eps) -> None (layernorm.cu:111-131, pybind.cpp:17), as
    tinychat/models/llama.py:33-36 calls it; compared with the reference's kernel on the same tensors."""
    eng = P.engine()
    x, gamma = rmsnorm_ref_inputs(dtype, DEV)
    out = torch.empty_like(x)
    assert eng.layernorm_forward_cuda(x, gamma, out, 1e-6) is None
    torch.cuda.synchronize()
    want = torch.from_numpy(LO.rmsnorm(np64(x), np64(gamma), 1e-6, dt_name(dtype))).to(dtype).to(DEV)
    assert int(_ulps(out, want, dtype).max()) <= 1
    gold = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_kernels.npz"))
    idx = torch.from_numpy(gold[f"rms_{dt_name(dtype)}_idx"]).long()
    out_ref = torch.from_numpy(gold[f"rms_{dt_name(dtype)}_y"]).view(dtype)
    u = _ulps(out.cpu().reshape(-1)[idx], out_ref, dtype)
    assert int(u.max()) <= 1 and float((u > 0).float().mean()) < 2e-3
    with pytest.raises(RuntimeError):
        eng.layernorm_forward_cuda(x, gamma.float(), out, 1e-6)      # layernorm.cu:122
    with pytest.raises(RuntimeError):
        eng.layernorm_forward_cuda(x.float(), gamma.float(), out.float(), 1e-6)   # fp32 is not dispatched (:14-25)


def test_rmsnorm_fp16_clamp_and_zero_rows():
    """reduction.cuh:78-82: fp16 results are clamped to +-(65504 - 1000) instead of overflowing to inf; an all-zero
    row gives zeros (rsqrt(eps) * 0)."""
    n = 1024
    x = torch.zeros(3, n, dtype=torch.float16, device=DEV)
    x[0, :] = 1.0
    x[2, 5] = 3.0
    gamma = torch.full((n,), 65000.0, dtype=torch.float16, device=DEV)
    y = _rmsnorm_abi(x, gamma, 1e-6)
    torch.cuda.synchronize()
    assert torch.isfinite(y).all()
    assert float(y[0, 0]) == float(torch.tensor(65504.0 - 1000.0).half())
    assert torch.count_nonzero(y[1]) == 0
    assert float(y[2, 5]) == float(torch.tensor(65504.0 - 1000.0).half()) and torch.count_nonzero(y[2]) == 1


def test_rmsnorm_under_graph_replay_in_a_chain():
    """norm -> GEMV -> norm captured in one CUDA graph with programmatic dependent launch: the norm reads its input
    only after the producer finished, and the GEMV after the norm."""
    dtype, H = torch.float16, 4096
    qw, s, z = gen_layer(H, H, dtype, seed=11, device=DEV)
    gamma = (1.0 + 0.1 * gen_x(1, H, dtype, seed=12, device=DEV)).view(H)
    x0 = gen_x(1, H, dtype, seed=13, device=DEV)
    eng = P.engine()
    a, c = torch.empty_like(x0), torch.empty_like(x0)

    def chain():
        eng.layernorm_forward_cuda(x0.view(1, 1, H), gamma, a.view(1, 1, H), 1e-5)
        b = eng.gemv_forward_cuda_new(a, qw, s, z, 1, H, H, 128)
        eng.layernorm_forward_cuda(b.view(1, 1, H), gamma, c.view(1, 1, H), 1e-5)
        return b
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        chain()
    side.synchronize()
    want_c = c.clone()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        chain()
    for _ in range(4):
        a.zero_(), c.zero_()
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(c, want_c)
    n1 = LO.rmsnorm(np64(x0), np64(gamma), 1e-5, "f16")
    assert rel_err(np64(a), n1) < 1e-3


# ------------------------------------------------------------------ fused gate + up + SiLU * mul (SURVEY.md §8f-1)
def _mlp_front_abi(x, gate, up, M, N, K, dtype, ws=True):
    y = torch.empty(M, N, dtype=dtype, device=DEV)
    lib = P.lib()
    nbytes = lib.b200awq_w4a16_mlp_front_workspace_bytes(M, N, K)
    w = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=DEV) if ws else None
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    rc = lib.b200awq_w4a16_mlp_front(p(x), p(gate[0]), p(gate[1]), p(gate[2]), p(up[0]), p(up[1]), p(up[2]), p(y), M, N, K, 128,
                                     0 if dtype == torch.float16 else 1, p(w) if ws else None, nbytes if ws else 0,
                                     ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    return rc, y


def _mlp_oracle(x, gate, up, dtype, rows=None):
    tr = lambda t: (t[0].cpu().numpy(), np64(t[1]), np64(t[2]))
    return LO.mlp_front(np64(x), tr(gate), tr(up), dtype=dt_name(dtype), rows=rows)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("N,K,M", [(N, K, M) for (N, K) in [(2816, 1024), (14336, 4096), (4608, 11008)]
                                   for M in (1, 4, 7, 8, 64, 2048) if not (M == 2048 and K == 11008)])   # keeps the oracle's float64 matmul short
def test_mlp_front_vs_oracle(N, K, M, dtype):
    """One fp16 token: the one-kernel path; everything else: two products + the elementwise kernel.  Against the oracle's
    composition with the reference's roundings; the product of two rounded factors is within 2 ulp of T normwise."""
    gate, up = gen_layer(N, K, dtype, seed=N + 1, device=DEV), gen_layer(N, K, dtype, seed=N + 2, device=DEV)
    x = (gen_x(M, K, dtype, seed=M + 5, device=DEV) * 0.5).contiguous()
    rc, y = _mlp_front_abi(x, gate, up, M, N, K, dtype)
    assert rc == 0, P.lib().b200awq_strerror(rc)
    torch.cuda.synchronize()
    rows = np.arange(0, N, 1 if M <= 8 and N < 4000 else 37)
    want = _mlp_oracle(x, gate, up, dtype, rows=rows)
    tol = 1.5e-3 if dtype == torch.float16 else 8e-3
    assert rel_err(np64(y[:, rows]), want) < tol


@pytest.mark.parametrize("split", [1, 2, 4])
@pytest.mark.parametrize("N,K", [(40, 512), (600, 4096), (2376, 4224), (14336, 4096)])
def test_mlp_front_one_token_kernel_equals_composition_bit_for_bit(N, K, split):
    """The fused kernel sums each product in exactly the order the plain decode kernel does and applies the same
    roundings: its output equals silu(gemv(gate)) * gemv(up) evaluated with torch on the plugin's GEMV results, up to
    the last place of expf (a handful of elements may differ by one ulp)."""
    dtype = torch.float16
    os.environ["B200AWQ_DECODE_SPLIT"] = str(split)
    P.lib().b200awq_reload_config()
    try:
        gate, up = gen_layer(N, K, dtype, seed=3, device=DEV), gen_layer(N, K, dtype, seed=4, device=DEV)
        x = gen_x(1, K, dtype, seed=8, device=DEV)
        rc, y = _mlp_front_abi(x, gate, up, 1, N, K, dtype, ws=False)     # the one-kernel path needs no workspace
        assert rc == 0, P.lib().b200awq_strerror(rc)
        eng = P.engine()
        g = eng.gemv_forward_cuda_new(x, *gate, 1, N, K, 128)
        u = eng.gemv_forward_cuda_new(x, *up, 1, N, K, 128)
        want = torch.nn.functional.silu(g) * u
        torch.cuda.synchronize()
        ulp = _ulps(y, want, dtype)
        assert int(ulp.max()) <= 1 and float((ulp > 0).float().mean()) < 5e-3
        assert rel_err(np64(y), _mlp_oracle(x, gate, up, dtype)) < 1.5e-3
    finally:
        os.environ.pop("B200AWQ_DECODE_SPLIT")
        P.lib().b200awq_reload_config()


def test_mlp_front_plugin_and_module_mirror():
    """awq_inference_engine.mlp_front_forward_cuda and llm_awq_b200.fused_mlp.QuantLlamaMLP (mirror of
    tinychat/modules/fused_mlp.py:11-83): shapes [1, tokens, hidden], both token regimes, workspace handled by the shim."""
    from llm_awq_b200.fused_mlp import QuantLlamaMLP
    dtype, H, I = torch.float16, 1024, 2816

    def wq(K, N, seed):
        m = P.WQLinear(4, 128, K, N, False, DEV)
        m.qweight, m.scales, m.scaled_zeros = gen_layer(N, K, dtype, seed=seed, device=DEV)
        return m
    gate, up, down = wq(H, I, 31), wq(H, I, 32), wq(I, H, 33)
    mlp = QuantLlamaMLP(gate, down, up)
    assert {"gate_proj_qweight", "gate_proj_scales", "gate_proj_scaled_zeros", "up_proj_qweight", "up_proj_scales",
            "up_proj_scaled_zeros"} <= set(mlp.state_dict().keys())
    for tokens in (1, 5, 40):
        x = (gen_x(tokens, H, dtype, seed=tokens, device=DEV) * 0.5).view(1, tokens, H)
        c = mlp.our_llama_mlp(x)
        torch.cuda.synchronize()
        assert c.shape == (1, tokens, I)
        want = _mlp_oracle(x.view(tokens, H), (gate.qweight, gate.scales, gate.scaled_zeros),
                           (up.qweight, up.scales, up.scaled_zeros), dtype)
        assert rel_err(np64(c.view(tokens, I)), want) < 1.5e-3
        y = mlp(x)
        assert y.shape == (1, tokens, H) and torch.isfinite(y).all()
    with pytest.raises(RuntimeError):
        P.engine().mlp_front_forward_cuda(x.float(), gate.qweight, gate.scales, gate.scaled_zeros, up.qweight, up.scales,
                                          up.scaled_zeros)


def test_mlp_front_rejects_bad_arguments():
    lib = P.lib()
    a = torch.zeros(64, dtype=torch.float16, device=DEV)
    p = ctypes.c_void_p(a.data_ptr())
    args = lambda m, n, k, g, dt, ws, wsb: (p, p, p, p, p, p, p, p, m, n, k, g, dt, ws, wsb, None)
    assert lib.b200awq_w4a16_mlp_front(*args(1, 4096, 4096, 64, 0, None, 0)) == -2      # group
    assert lib.b200awq_w4a16_mlp_front(*args(1, 4096, 4096, 128, 5, None, 0)) == -4     # dtype
    assert lib.b200awq_w4a16_mlp_front(*args(1, 4100, 4096, 128, 0, None, 0)) == -1     # n % 8
    assert lib.b200awq_w4a16_mlp_front(*args(16, 4104, 4096, 128, 0, p, 1 << 30)) == -1  # n % 128 from 8 tokens
    assert lib.b200awq_w4a16_mlp_front(*args(4, 4096, 4096, 128, 0, None, 0)) == -6     # workspace required beyond one token
    assert lib.b200awq_w4a16_mlp_front_workspace_bytes(4, 4096, 4096) == 2 * 4 * 4096 * 2
