"""CPU-side checks: host mirror vs the reference-generated goldens, ABI surface, no fallback."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import llm_awq_b200 as P
from oracle import w4a16_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = np.load(os.path.join(ROOT, "tests", "golden", "reference_packer.npz"))


@pytest.mark.parametrize("idx", range(6))
def test_host_packer_matches_reference(idx):
    q = torch.from_numpy(G[f"pack{idx}_q"].astype(np.int32))
    packed = P.pack_intweight(q, interleave=4, kstride=64)
    assert packed.dtype == torch.int16
    assert np.array_equal(packed.numpy(), G[f"pack{idx}_packed"])
    assert torch.equal(P.unpack_intweight(packed).to(torch.int32), q)


def test_zeros_width_and_buffer_shapes():
    for i, a, b in zip(G["zw_in"], G["zw_g128"], G["zw_g64"]):
        assert P.calculate_zeros_width(int(i), 128) == a and P.calculate_zeros_width(int(i), 64) == b
    for K, N, qr, qc, sr, sc, zr, zc in G["init_shapes"]:
        m = P.WQLinear(4, 128, int(K), int(N), False, "cpu")
        assert tuple(m.qweight.shape) == (qr, qc) and m.qweight.dtype == torch.int16
        assert tuple(m.scales.shape) == (sr, sc) and tuple(m.scaled_zeros.shape) == (zr, zc)
        assert set(m.state_dict().keys()) == {"qweight", "scales", "scaled_zeros"}


@pytest.mark.parametrize("tag,dt", [("f32", torch.float32), ("f16", torch.float16), ("bf16", torch.bfloat16)])
def test_from_linear_matches_reference(tag, dt):
    N, K = G[f"fl_{tag}_wdq"].shape
    lin = torch.nn.Linear(K, N, bias=True)
    lin.weight.data = torch.from_numpy(G[f"fl_{tag}_wdq"]).to(dt)
    lin.bias.data = torch.from_numpy(G[f"fl_{tag}_bias"]).to(dt)
    lin = lin.to(dt)
    scales = torch.from_numpy(G[f"fl_{tag}_scales"]).to(dt)
    zeros = torch.from_numpy(G[f"fl_{tag}_zeros"]).to(dt)
    m = P.WQLinear.from_linear(lin, 4, 128, False, scales, zeros)
    assert np.array_equal(m.qweight.numpy(), G[f"fl_{tag}_qweight"])
    assert np.array_equal(m.scales.float().numpy(), G[f"fl_{tag}_sbuf"])
    assert np.array_equal(m.scaled_zeros.float().numpy(), G[f"fl_{tag}_zbuf"])
    assert np.array_equal(m.bias.detach().float().numpy(), G[f"fl_{tag}_bias"])
    empty = P.WQLinear.from_linear(lin, 4, 128, init_only=True)
    assert int(empty.qweight.abs().sum()) == 0


def test_constructor_rejects_like_reference():
    with pytest.raises(NotImplementedError):
        P.WQLinear(8, 128, 256, 64, False, "cpu")
    with pytest.raises(AssertionError):
        P.WQLinear(4, 128, 200, 64, False, "cpu")
    with pytest.raises(AssertionError):
        P.WQLinear(4, 128, 256, 60, False, "cpu")
    m = P.WQLinear(4, -1, 256, 64, True, "cpu")
    assert m.group_size == 256 and m.bias is not None


def test_abi_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "b200awq.h")).read()
    names = set(re.findall(r"^\s*(?:int|size_t|unsigned long long|const char\*)\s+(\w+)\s*\(", hdr, flags=re.M))
    assert {"b200awq_w4a16_gemv", "b200awq_w4a16_gemm", "b200awq_w4a16_gemm_workspace_bytes", "gemv_forward_4bit",
            "gemm_forward_4bit", "b200awq_set_pdl", "b200awq_launch_count", "b200awq_strerror",
            "b200awq_version"} <= names
    lib = P.lib()
    for n in names:
        assert hasattr(lib, n), n
    assert lib.b200awq_version().startswith(b"b200awq")
    assert lib.b200awq_w4a16_gemm_workspace_bytes(2048, 4096, 4096) == 0
    assert b"group" in lib.b200awq_strerror(-2)


def test_abi_rejects_bad_arguments_without_a_gpu():
    """Argument validation happens before anything touches the device."""
    lib = P.lib()
    buf = (ctypes.c_char * 64)()
    a = ctypes.c_void_p((ctypes.addressof(buf) + 15) & ~15)
    args = lambda m, n, k, g, dt: (a, a, a, a, a, m, n, k, g, dt, None)
    assert lib.b200awq_w4a16_gemv(*args(1, 4096, 4096, 64, 0)) == -2      # group
    assert lib.b200awq_w4a16_gemv(*args(1, 4096, 4096, 128, 7)) == -4     # dtype
    assert lib.b200awq_w4a16_gemv(*args(1, 4100, 4096, 128, 0)) == -1     # n % 8
    assert lib.b200awq_w4a16_gemv(*args(1, 4096, 4000, 128, 0)) == -1     # k % 128
    assert lib.b200awq_w4a16_gemv(None, a, a, a, a, 1, 4096, 4096, 128, 0, None) == -3   # null pointer
    off = ctypes.c_void_p(a.value + 2)
    assert lib.b200awq_w4a16_gemv(off, a, a, a, a, 1, 4096, 4096, 128, 0, None) == -3    # misaligned
    if not torch.cuda.is_available():
        rc = lib.b200awq_w4a16_gemv(*args(8, 4096, 4096, 128, 0))
        assert rc != 0  # no device (or batch) -> error, never a silent CPU path


def test_extension_surface_and_no_cpu_fallback():
    eng = P.engine()
    assert eng.__name__ == "awq_inference_engine"
    assert callable(eng.gemv_forward_cuda_new) and callable(eng.gemm_forward_cuda_new)
    import awq_inference_engine  # what the reference's qmodule.py:4 does
    assert awq_inference_engine is eng
    m = P.WQLinear(4, 128, 256, 64, False, "cpu")
    with pytest.raises(RuntimeError):
        m(torch.zeros(1, 256, dtype=torch.float16))      # CPU tensors are rejected, not computed on the host
    with pytest.raises(RuntimeError):
        m(torch.zeros(9, 256, dtype=torch.float16))


def test_oracle_is_not_imported_by_the_product():
    pkg = os.path.join(ROOT, "llm_awq_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                assert "oracle" not in open(os.path.join(dirpath, f)).read().replace("test oracle", ""), f


def test_unmodified_reference_wqlinear_binds_to_this_engine():
    """The reference's own qmodule.py does `import awq_inference_engine` (qmodule.py:4): with our plugin
    directory on sys.path that import must pick up THIS build; the drop-in WQLinear must hold the buffers the reference's
    WQLinear holds (stored in tests/golden/reference_callsites.npz; the reference's code does not run here), and its
    forward must reach our entry points (which reject CPU tensors instead of computing on the host)."""
    import importlib
    import sys
    P.install()
    sys.modules.pop("awq_inference_engine", None)
    eng = importlib.import_module("awq_inference_engine")
    assert os.path.abspath(eng.__file__).startswith(P.install())
    gold = np.load(os.path.join(ROOT, "tests", "golden", "reference_callsites.npz"))
    want = {k[len("state_"):-len("_shape")]: (tuple(gold[k]), str(gold[k[:-len("_shape")] + "_dtype"]))
            for k in gold.files if k.startswith("state_") and k.endswith("_shape")}
    m = P.WQLinear(4, 128, 256, 64, False, "cpu")
    assert {k: (tuple(v.shape), str(v.dtype)) for k, v in m.state_dict().items()} == want
    for tokens in (1, 9):      # GEMV branch and GEMM branch of the reference's forward (qmodule.py:206-220)
        with pytest.raises(RuntimeError, match="CUDA"):
            m(torch.zeros(tokens, 256, dtype=torch.float16))


def test_packer_out_of_range_and_raw_weight_from_linear_match_reference():
    """Unmasked OR of out-of-range integers (reference qmodule.py:50-55) is reproduced bit for bit."""
    q = torch.from_numpy(G["packoob_q"])
    assert np.array_equal(P.pack_intweight(q).numpy(), G["packoob_packed"])
    assert np.array_equal(O.pack_intweight(G["packoob_q"]), G["packoob_packed"])
    for tag, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
        N, K = G[f"flraw_{tag}_w"].shape
        lin = torch.nn.Linear(K, N, bias=False)
        lin.weight.data = torch.from_numpy(G[f"flraw_{tag}_w"]).to(dt)
        lin = lin.to(dt)
        m = P.WQLinear.from_linear(lin, 4, 128, False, torch.from_numpy(G[f"flraw_{tag}_scales"]).to(dt),
                                   torch.from_numpy(G[f"flraw_{tag}_zeros"]).to(dt))
        assert np.array_equal(m.qweight.numpy(), G[f"flraw_{tag}_qweight"])
        assert np.array_equal(m.scales.float().numpy(), G[f"flraw_{tag}_sbuf"])
        assert np.array_equal(m.scaled_zeros.float().numpy(), G[f"flraw_{tag}_zbuf"])
        qw, sbuf, zbuf = O.from_linear(G[f"flraw_{tag}_w"], G[f"flraw_{tag}_scales"], G[f"flraw_{tag}_zeros"], 128, tag)
        assert np.array_equal(qw, G[f"flraw_{tag}_qweight"])
