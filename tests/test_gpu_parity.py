"""GPU parity tests proper: the sm_100a kernels, called through the C ABI (ctypes, raw device
pointers) and through the `awq_inference_engine` extension, against the CPU oracle.

Tolerances (BASELINE.json north_star: "within 1e-3 relative"):
  * fp16:  ||y - Y64|| / ||Y64|| <= 1e-3 against the exact (float64) oracle; the kernels accumulate
    in fp32 so the measured error is the output rounding (~3e-4).
  * bf16:  the output rounding alone is ~1.6e-3 normwise, so the check is against the oracle ROUNDED
    to bf16: ||y - rn_bf16(Y64)|| / ||Y64|| <= 1e-3 (a few elements may land one ulp off).
  * one-hot activations read back a dequantised weight column: BIT-EXACT against the oracle's w~.
"""
import ctypes

import numpy as np
import pytest
import torch

import llm_awq_b200 as P
from oracle import w4a16_oracle as O
from awq_testutil import abi_call, dt_name, gen_layer, gen_x, np64, oracle_forward, rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-3
DTYPES = [torch.float16, torch.bfloat16]


def check(y, ref, dtype, tol=TOL):
    y = np64(y)
    assert np.isfinite(y).all()
    if dtype == torch.bfloat16:
        ref_r = O.rn_bf16(ref)
        err = float(np.linalg.norm(y - ref_r) / np.linalg.norm(ref))
    else:
        err = rel_err(y, ref)
    assert err <= tol, err
    return err


# ------------------------------------------------------------------ decode path (GEMV ABI)
@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("M", [1, 2, 3, 4, 5, 6, 7])
@pytest.mark.parametrize("N,K", [(8, 128), (24, 256), (64, 384), (512, 1024), (4096, 4096)])
def test_gemv_abi_vs_oracle(N, K, M, dtype):
    qw, s, z = gen_layer(N, K, dtype, seed=N + K, device=DEV)
    x = gen_x(M, K, dtype, seed=M, device=DEV)
    rc, y = abi_call(P.lib(), x, qw, s, z, M, N, K, dtype, "gemv")
    assert rc == 0, P.lib().b200awq_strerror(rc)
    torch.cuda.synchronize()
    check(y, oracle_forward(x, qw, s, z, dtype), dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("N,K", [(6144, 4096), (14336, 4096), (4096, 14336), (4096, 11008), (1280, 8192), (8192, 3584)])
def test_gemv_model_shapes(N, K, dtype):
    """Llama-3-8B / Llama-2-7B / 70B-TP8 layer shapes (SURVEY.md §8d), incl. padded scale rows."""
    qw, s, z = gen_layer(N, K, dtype, seed=7, device=DEV)
    x = gen_x(1, K, dtype, seed=3, device=DEV)
    rc, y = abi_call(P.lib(), x, qw, s, z, 1, N, K, dtype, "gemv")
    assert rc == 0
    rows = np.arange(0, N, 7)
    check(y[:, rows], oracle_forward(x, qw, s, z, dtype, rows=rows), dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("M", [3, 4])
@pytest.mark.parametrize("N,K", [(6144, 4096), (4096, 14336), (4096, 11008), (8192, 3584)])
def test_gemv_model_shapes_batch_sweep(N, K, M, dtype):
    """BASELINE configs[4] (bs = 4): 3-4 tokens take k unsplit up to 4096 per CTA in the streaming kernel and the
    tcgen05 skinny kernel when k > 8192 (api.cu use_flat); both routes against the oracle on the model shapes."""
    qw, s, z = gen_layer(N, K, dtype, seed=17, device=DEV)
    x = gen_x(M, K, dtype, seed=5, device=DEV)
    rc, y = abi_call(P.lib(), x, qw, s, z, M, N, K, dtype, "gemv")
    assert rc == 0
    rows = np.arange(0, N, 11)
    check(y[:, rows], oracle_forward(x, qw, s, z, dtype, rows=rows), dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("kind,M", [("gemv", 1), ("gemv", 5), ("gemm", 1), ("gemm", 12), ("gemm", 40), ("gemm", 300)])
def test_one_hot_reads_back_dequantised_weight_bit_exact(kind, M, dtype):
    N, K = 256, 512
    qw, s, z = gen_layer(N, K, dtype, seed=11, device=DEV)
    ks = [(37 * i + 5) % K for i in range(M)]
    x = torch.zeros(M, K, dtype=dtype, device=DEV)
    for i, k in enumerate(ks):
        x[i, k] = 1.0
    rc, y = abi_call(P.lib(), x, qw, s, z, M, N, K, dtype, kind)
    assert rc == 0
    w = O.dequant_weight(qw.cpu().numpy(), np64(s), np64(z), 128, dt_name(dtype))   # [N, K]
    assert np.array_equal(np64(y), w[:, ks].T)


# ------------------------------------------------------------------ prefill / batched path (GEMM ABI)
@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("M", [1, 7, 8, 9, 16, 17, 31, 33, 64, 100, 128, 192, 193, 256, 300, 513])
def test_gemm_abi_vs_oracle_small(M, dtype):
    N, K = 384, 512
    qw, s, z = gen_layer(N, K, dtype, seed=M, device=DEV)
    x = gen_x(M, K, dtype, seed=M + 1, device=DEV)
    rc, y = abi_call(P.lib(), x, qw, s, z, M, N, K, dtype, "gemm")
    assert rc == 0, P.lib().b200awq_strerror(rc)
    check(y, oracle_forward(x, qw, s, z, dtype), dtype)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("M,N,K", [(2048, 4096, 4096), (2048, 6144, 4096), (2048, 4096, 14336), (777, 14336, 4096),
                                   (64, 4096, 4096), (16, 4096, 11008), (2048, 1280, 8192)])
def test_gemm_full_size_spot_rows(M, N, K, dtype):
    qw, s, z = gen_layer(N, K, dtype, seed=5, device=DEV)
    x = gen_x(M, K, dtype, seed=6, device=DEV)
    rc, y = abi_call(P.lib(), x, qw, s, z, M, N, K, dtype, "gemm")
    assert rc == 0
    rows = np.concatenate([np.arange(0, N, 61), np.arange(N - 130, N)])
    check(y[:, rows], oracle_forward(x, qw, s, z, dtype, rows=rows), dtype)


def test_gemm_linearity_and_determinism_full_size():
    """Size-independent properties at BASELINE's full prefill size."""
    M, N, K = 2048, 4096, 4096
    dtype = torch.float16
    qw, s, z = gen_layer(N, K, dtype, seed=1, device=DEV)
    x = gen_x(M, K, dtype, seed=2, device=DEV)
    _, y1 = abi_call(P.lib(), x, qw, s, z, M, N, K, dtype, "gemm")
    _, y2 = abi_call(P.lib(), x, qw, s, z, M, N, K, dtype, "gemm")
    assert torch.equal(y1, y2)                                  # no atomics, fixed reduction order
    _, yh = abi_call(P.lib(), (x * 2).contiguous(), qw, s, z, M, N, K, dtype, "gemm")
    big = y1.abs() > 2.0 ** -13                                  # fp16 subnormal outputs lose a bit when halved
    assert torch.equal(yh.float()[big], y1.float()[big] * 2)    # scaling by 2 is exact in fp16 / fp32 (no overflow here)
    # rows of the batch are independent: a token computed alone through the decode path agrees
    _, y_row = abi_call(P.lib(), x[1000:1001].contiguous(), qw, s, z, 1, N, K, dtype, "gemv")
    assert rel_err(np64(y_row), np64(y1[1000:1001])) < 5e-4


# ------------------------------------------------------------------ extension + module (the reference's call sites)
@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
def test_wqlinear_module_dispatch_and_bias(dtype):
    torch.manual_seed(0)
    K, N = 512, 256
    lin = torch.nn.Linear(K, N, bias=True).to(dtype)
    w = lin.weight.data.float()
    sc, zp = O.pseudo_quantize_scales_zeros(w.numpy(), 128)
    scales, zeros = torch.from_numpy(sc).to(dtype), torch.from_numpy(zp).to(dtype)
    m = P.WQLinear.from_linear(lin, 4, 128, False, scales, zeros).to(DEV)
    for shape in [(1, 1, K), (1, 7, K), (2, 4, K), (1, 33, K), (3, 100, K)]:
        x = torch.randn(*shape, dtype=dtype, device=DEV)
        y = m(x)
        assert y.shape == (*shape[:-1], N) and y.dtype == dtype
        ref = O.wq_linear_forward(np64(x), m.qweight.cpu().numpy(), np64(m.scales), np64(m.scaled_zeros),
                                  bias=np64(m.bias), dtype=dt_name(dtype))
        tol = 1e-3 if dtype == torch.float16 else 6e-3   # bias add is a second bf16 rounding in PyTorch
        assert rel_err(np64(y), ref) < tol
    # and the quantised layer approximates the dense one (4-bit error, sanity only)
    x = torch.randn(4, K, dtype=dtype, device=DEV)
    dense = torch.nn.functional.linear(x.float(), lin.weight.float().to(DEV), lin.bias.float().to(DEV))
    assert rel_err(np64(m(x)), np64(dense)) < (0.2 if dtype == torch.float16 else 0.35)   # the reference's bf16 quantiser arithmetic is this lossy


def test_engine_signatures_errors_and_streams():
    eng = P.engine()
    N, K = 256, 512
    qw, s, z = gen_layer(N, K, torch.float16, device=DEV)
    x = gen_x(3, K, torch.float16, device=DEV)
    y = eng.gemv_forward_cuda_new(x.view(1, 3, K), qw, s, z, 3, N, K, 128)
    assert y.shape == (1, 3, N)
    y2 = eng.gemm_forward_cuda_new(x.view(3, 1, K), qw, s, z)
    assert y2.shape == (3, 1, N) and torch.equal(y.view(3, N), y2.view(3, N))
    with pytest.raises(RuntimeError):                      # reference: gemv_cuda.cu:329
        eng.gemv_forward_cuda_new(gen_x(8, K, device=DEV), qw, s, z, 8, N, K, 128)
    with pytest.raises(RuntimeError):                      # reference: gemv_cuda.cu:334
        eng.gemv_forward_cuda_new(x, qw, s, z, 3, N, K, 64)
    with pytest.raises(RuntimeError):                      # dtype mismatch, gemv_cuda.cu:260
        eng.gemv_forward_cuda_new(x, qw, s.bfloat16(), z, 3, N, K, 128)
    with pytest.raises(RuntimeError):
        eng.gemm_forward_cuda_new(x.float(), qw, s, z)     # dispatch_utils.cuh:13-17
    # side stream + CUDA graph capture/replay (no allocation or sync inside the C ABI)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        y3 = eng.gemv_forward_cuda_new(x, qw, s, z, 3, N, K, 128)
    st.synchronize()
    assert torch.equal(y3, y.view(3, N))
    g = torch.cuda.CUDAGraph()
    xs = x.clone()
    with torch.cuda.graph(g):
        yg = eng.gemv_forward_cuda_new(xs, qw, s, z, 3, N, K, 128)
        yg2 = eng.gemm_forward_cuda_new(xs, qw, s, z)
    xs.copy_(x * 2)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(yg.float(), y.view(3, N).float() * 2) and torch.equal(yg, yg2)
    before = eng.launch_count()
    eng.gemm_forward_cuda_new(x, qw, s, z)
    assert eng.launch_count() == before + 1


def test_abi_error_codes_on_device():
    lib = P.lib()
    N, K = 256, 512
    qw, s, z = gen_layer(N, K, torch.float16, device=DEV)
    x = gen_x(8, K, torch.float16, device=DEV)
    assert abi_call(lib, x, qw, s, z, 8, N, K, torch.float16, "gemv")[0] == -5
    qw2, s2, z2 = gen_layer(72, K, torch.float16, device=DEV)
    assert abi_call(lib, x, qw2, s2, z2, 8, 72, K, torch.float16, "gemm")[0] == -1     # gemm needs n % 128 == 0
    assert abi_call(lib, x[:1], qw2, s2, z2, 1, 72, K, torch.float16, "gemv")[0] == 0  # gemv only n % 8


# ------------------------------------------------------------------ against the reference's own kernels (sm_100a rebuild)
REF_KERNEL_CASES = [(1, 4096, 4096), (4, 6144, 4096), (7, 4096, 14336), (16, 4096, 4096),
                    (64, 14336, 4096), (192, 4096, 4096), (193, 4096, 4096), (2048, 4096, 4096)]


def ref_kernel_rows(M):
    """Rows of the output kept in tests/golden/reference_kernels.npz: all of them up to 16, else 16 seeded ones."""
    return np.arange(M) if M <= 16 else np.sort(np.random.default_rng(M).choice(M, 16, replace=False))


@pytest.fixture(scope="module")
def ref_kernels():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_kernels.npz"))


@pytest.mark.parametrize("dtype", DTYPES, ids=["f16", "bf16"])
@pytest.mark.parametrize("M,N,K", REF_KERNEL_CASES)
def test_matches_reference_kernels(ref_kernels, M, N, K, dtype):
    """Same packed inputs as the reference kernels rebuilt for sm_100a were given (their outputs are stored by
    tests/golden/make_golden.py --kernels): 1e-3 normwise (the reference accumulates in fp16, so it is the LESS
    accurate of the two vs the oracle)."""
    eng = P.engine()
    qw, s, z = gen_layer(N, K, dtype, seed=9, device=DEV)
    x = (gen_x(M, K, dtype, seed=10, device=DEV) * 0.25).contiguous()   # keep fp16 chains away from overflow
    key = f"w4_{M}x{N}x{K}_{dt_name(dtype)}"
    assert float(np64(x).sum()) == float(ref_kernels[key + "_xsum"])       # the inputs the reference was given
    assert int(qw.cpu().numpy().astype(np.int64).sum()) == int(ref_kernels[key + "_qwsum"])
    if M < 8:
        y = eng.gemv_forward_cuda_new(x, qw, s, z, M, N, K, 128)
    else:
        y = eng.gemm_forward_cuda_new(x, qw, s, z)
    torch.cuda.synchronize()
    cols = np.arange(0, N, 37)
    y64 = oracle_forward(x, qw, s, z, dtype, rows=cols)
    e_ours = rel_err(np64(y[:, cols]), y64)             # every row, every 37th column
    # the stored reference sample: up to 16 rows at every 74th column
    rows, sub = ref_kernel_rows(M), slice(None, None, 2)
    y_ref = np64(torch.from_numpy(ref_kernels[key + "_y"]).view(dtype))
    ys, y64s = np64(y[:, cols[sub]])[rows], y64[rows][:, sub]
    e_ours_s = rel_err(ys, y64s)
    e_ref = rel_err(y_ref, y64s)
    e_mut = rel_err(ys, y_ref)
    print(f"M={M} N={N} K={K} {dt_name(dtype)}: ours-vs-oracle {e_ours:.2e} (sample {e_ours_s:.2e})  "
          f"ref-vs-oracle {e_ref:.2e}  ours-vs-ref {e_mut:.2e}")
    lim = 1e-3 if dtype == torch.float16 else 4e-3      # bf16: two independently rounded bf16 outputs
    assert e_ours <= lim
    assert e_mut <= max(lim, 2 * e_ref)
    assert e_ours_s <= e_ref * 1.05 + 1e-6              # never less accurate than the reference
