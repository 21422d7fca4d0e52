"""Generate tests/golden/*.npz by running the REFERENCE's own Python on CPU.

Needs a checkout of the reference (its path in AWQ_REFERENCE) and a built package:

    python tests/golden/make_golden.py

reference_kernels.npz is made on a GPU from the reference's kernels instead (kernels_golden).

The reference module ``awq.quantize.qmodule`` does ``import awq_inference_engine`` at
import time (qmodule.py:4); a stub module is registered for that name because only the
pure-PyTorch / numpy packer code is exercised here (no kernel is called).
The fixtures pin oracle/w4a16_oracle.py (pack layout, buffer shapes, from_linear,
quantiser formulas); the reference has no golden vectors of its own (SURVEY.md §4).
"""
import os
import sys
import types

import numpy as np
import torch

REF = os.environ.get("AWQ_REFERENCE", "/root/reference")
HERE = os.path.dirname(os.path.abspath(__file__))


def _import_reference():
    sys.modules.setdefault("awq_inference_engine", types.ModuleType("awq_inference_engine"))
    # awq/quantize/__init__.py pulls in w8a8_linear / smooth; import the two files directly
    import importlib.util

    def load(name, rel):
        spec = importlib.util.spec_from_file_location(name, os.path.join(REF, rel))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    qmodule = load("ref_qmodule", "awq/quantize/qmodule.py")
    # quantizer.py has package-relative imports at module top; extract the one function
    src = open(os.path.join(REF, "awq/quantize/quantizer.py")).read()
    start = src.index("def pseudo_quantize_tensor(")
    end = src.index("@torch.no_grad()", start)
    ns = {"torch": torch}
    exec(compile(src[start:end], "ref_quantizer_excerpt", "exec"), ns)
    return qmodule, ns["pseudo_quantize_tensor"]


def _import_repacker():
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_repacker", os.path.join(REF, "tinychat/offline-weight-repacker.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def repacker_golden():
    """tests/golden/reference_repacker.npz: v1 tensors and what the reference's offline repacker makes of them
    (tinychat/offline-weight-repacker.py:8-79), for llm_awq_b200/repack.py."""
    rp = _import_repacker()
    g = torch.Generator().manual_seed(77)
    out = {}
    for idx, (N, K, G) in enumerate([(8, 128, 128), (16, 256, 128), (64, 1024, 128), (32, 2048, 128)]):
        qw = torch.randint(-2 ** 31, 2 ** 31 - 1, (N, K // 8), generator=g, dtype=torch.int64).to(torch.int32)
        ng = K // G
        scales = (0.004 + 0.012 * torch.rand(N, ng, generator=g)).half()
        qz = torch.randint(-2 ** 31, 2 ** 31 - 1, (N, -(-ng // 8)), generator=g, dtype=torch.int64).to(torch.int32)
        out[f"r{idx}_qweight_v1"] = qw.numpy()
        out[f"r{idx}_scales_v1"] = scales.float().numpy()
        out[f"r{idx}_qzeros_v1"] = qz.numpy()
        out[f"r{idx}_unpacked"] = rp.qweight_unpack(qw).numpy().astype(np.uint8)
        out[f"r{idx}_qweight_v2"] = rp.qweight_pack_v1_to_v2(qw, 4, 64).numpy()
        out[f"r{idx}_scaled_zeros"] = rp.multiply_scale_qzero_negative(scales, qz, zp_shift=-8).float().numpy()
    np.savez_compressed(os.path.join(HERE, "reference_repacker.npz"), **out)
    print("wrote reference_repacker.npz", len(out), "arrays")


def layer_ops_golden():
    """tests/golden/reference_layer_ops.npz: what the reference's own PYTHON statements of the ops around the linears
    give on CPU -- for oracle/layer_oracle.py.  The kernels themselves are CUDA-only; these are the definitions the
    reference keeps beside them:
      * RMSNorm._norm * weight                       tinychat/models/llama.py:24-31
      * precompute_freqs_cis + apply_rotary_emb      tinychat/models/llama.py:39-47, 68-84 (pairs (i, i + d/2))
      * precompute_freqs                             tinychat/models/llama.py:50-57 (table for fused_rope_with_pos)
      * the KV-cache store and the softmax attention of the prefill branch
                                                     tinychat/modules/fused_attn.py:256-305 (restated below with the
                                                     same tensor expressions: the module itself needs CUDA caches)
    Inputs hold fp16-representable values; everything is computed in fp32 / fp64 and stored unrounded."""
    sys.modules.setdefault("awq_inference_engine", types.ModuleType("awq_inference_engine"))
    if REF not in sys.path:
        sys.path.insert(0, REF)
    import contextlib
    import math
    with contextlib.redirect_stdout(sys.stderr):
        import tinychat.models.llama as L
    g = torch.Generator().manual_seed(4242)
    out = {}
    # --- RMSNorm
    for idx, (rows, dim, eps) in enumerate([(3, 64, 1e-6), (5, 4096, 1e-5), (2, 200, 1e-6)]):
        x = torch.randn(rows, dim, generator=g).half().double() * 3
        w = (1 + 0.1 * torch.randn(dim, generator=g)).half().double()
        norm = L.RMSNorm(dim, eps=eps).double()
        with torch.no_grad():
            norm.weight.copy_(w)
            y = norm._norm(x) * norm.weight
        out[f"n{idx}_x"], out[f"n{idx}_w"], out[f"n{idx}_eps"], out[f"n{idx}_y"] = x.numpy(), w.numpy(), np.float64(eps), y.numpy()
    # --- RoPE + one decode step seen as the last row of a prefill
    for idx, (S, H, Hkv, D, theta, scale) in enumerate([(9, 4, 2, 16, 10000.0, 1.0), (17, 8, 8, 32, 500000.0, 0.5),
                                                         (12, 8, 2, 64, 10000.0, 1.0)]):
        xq = torch.randn(1, S, H, D, generator=g).half().float()
        xk = torch.randn(1, S, Hkv, D, generator=g).half().float()
        xv = torch.randn(1, S, Hkv, D, generator=g).half().float()
        fc = L.precompute_freqs_cis(D, S, theta, scale)
        rq, rk = L.apply_rotary_emb(xq, xk, freqs_cis=fc)
        # the table the callers hand to fused_rope_with_pos (llama.py:312-317 passes the scale, precompute_freqs :50-57
        # does not use it: the table is always unscaled) and what that table means in terms of apply_rotary_emb
        table = L.precompute_freqs(D, S, theta, scale)  # [S, 1, 1, D]
        rq1, rk1 = L.apply_rotary_emb(xq, xk, freqs_cis=L.precompute_freqs_cis(D, S, theta, 1.0))
        # cache store, fused_attn.py:262-270
        keys_store = rk.reshape(1, S, Hkv, D // 8, 8).permute(0, 2, 3, 1, 4).contiguous()   # [B, Hkv, D/8, S, 8]
        values_store = xv.transpose(2, 1).contiguous()                                       # [B, Hkv, S, D]
        # attention, fused_attn.py:290-304, fp32, causal: the last row sees every position
        rep = H // Hkv
        keys = torch.repeat_interleave(rk, dim=2, repeats=rep).transpose(1, 2)
        values = torch.repeat_interleave(xv, dim=2, repeats=rep).transpose(1, 2)
        q_ = rq.transpose(1, 2)
        scores = torch.matmul(q_.double(), keys.double().transpose(2, 3)) / math.sqrt(D)
        mask = torch.full((S, S), float("-inf")).triu(1).double()
        scores = torch.softmax(scores + mask, dim=-1)
        o = torch.matmul(scores, values.double()).transpose(1, 2)                            # [B, S, H, D]
        for k, v in dict(xq=xq, xk=xk, xv=xv, rq=rq, rk=rk, rq1=rq1, rk1=rk1, table=table.reshape(S, D), cache_k=keys_store,
                         cache_v=values_store, out=o).items():
            out[f"a{idx}_{k}"] = v.double().numpy()
        out[f"a{idx}_cfg"] = np.array([S, H, Hkv, D, theta, scale], dtype=np.float64)
    # --- the cos|sin table of the HF-attention branch (rotary_embedding_neox's input), fused_attn.py:25-59, and what the
    # rotation means in terms of apply_rotary_emb at the same positions
    with contextlib.redirect_stdout(sys.stderr):
        import tinychat.modules.fused_attn as FA
    for idx, (dim, maxpos, base, heads) in enumerate([(16, 64, 10000, 4), (64, 300, 10000, 3), (128, 512, 10000, 2)]):
        rot = FA.QuantLlamaRotaryEmbedding(dim, max_position_embeddings=maxpos, base=base, device="cpu")
        pos = torch.randint(0, maxpos, (11,), generator=g)
        pos[0], pos[1] = 0, maxpos - 1
        xq = torch.randn(1, 11, heads, dim, generator=g).half().float()
        xk = torch.randn(1, 11, heads, dim, generator=g).half().float()
        fc = L.precompute_freqs_cis(dim, maxpos, float(base), 1.0)[pos]
        rq, rk = L.apply_rotary_emb(xq, xk, freqs_cis=fc)
        out[f"c{idx}_cfg"] = np.array([dim, maxpos, base, heads], dtype=np.float64)
        out[f"c{idx}_cache"] = rot.cos_sin_cache.numpy()                   # float16
        out[f"c{idx}_pos"] = pos.numpy()
        for k, v in dict(xq=xq, xk=xk, rq=rq, rk=rk).items():
            out[f"c{idx}_{k}"] = v.double().numpy()
    np.savez_compressed(os.path.join(HERE, "reference_layer_ops.npz"), **out)
    print("wrote reference_layer_ops.npz", len(out), "arrays")


def mlp_callsite_golden():
    """tests/golden/reference_mlp_callsite.npz: the reference's own, unmodified ``QuantLlamaMLP.our_llama_mlp``
    (tinychat/modules/fused_mlp.py:36-83) EXECUTED on CPU.  Its two engine calls are served by a stub
    ``awq_inference_engine`` whose linears are the (separately pinned) W4A16 oracle rounded to fp16; everything the
    reference does around them -- which branch it takes, the zeros it passes (``- 8 * scales`` in the GEMM branch,
    :69,76), ``F.silu`` on the fp16 tensor, the fp16 product -- is the reference's code.  Pins
    oracle/layer_oracle.py::mlp_front (order and placement of the roundings)."""
    root = os.path.dirname(os.path.dirname(HERE))
    if root not in sys.path:
        sys.path.insert(0, root)
    from oracle import w4a16_oracle as O
    if REF not in sys.path:
        sys.path.insert(0, REF)
    qmodule, _ = _import_reference()
    eng = sys.modules["awq_inference_engine"]
    calls = []

    def linear(x, qw, s, z):
        y = O.wq_linear_forward(x.double().numpy(), qw.numpy(), s.double().numpy(), z.double().numpy(), dtype="f16")
        return torch.from_numpy(O.rn_f16(y)).to(torch.float16)

    def gemv(x, qw, s, z, m, n, k, g):
        calls.append(("gemv", m, n, k, g))
        return linear(x, qw, s, z)

    def gemm(x, qw, s, z):
        calls.append(("gemm", z.clone()))
        return linear(x, qw, s, z)
    eng.gemv_forward_cuda_new, eng.gemm_forward_cuda_new = gemv, gemm
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):
        import tinychat.modules.fused_mlp as FM
    g = torch.Generator().manual_seed(606)
    out = {}
    for idx, (N, K) in enumerate([(128, 256), (256, 128)]):
        def layer(n, k):
            m = qmodule.WQLinear(4, 128, k, n, False, "cpu")
            q = torch.randint(0, 16, (n, k), generator=g, dtype=torch.int32)
            m.qweight = qmodule.pack_intweight(q, interleave=4, kstride=64)
            ng = k // 128
            sc = (0.004 + 0.01 * torch.rand(ng, n, generator=g)).half()
            zz = torch.randint(0, 16, (ng, n), generator=g).half()
            m.scales[:ng] = sc
            m.scaled_zeros[:ng] = -(sc * zz)
            return m
        gate, up, down = layer(N, K), layer(N, K), layer(K, N)
        mlp = FM.QuantLlamaMLP(gate, down, up)
        for nm, mod in (("gate", gate), ("up", up)):
            out[f"m{idx}_{nm}_qweight"] = mod.qweight.numpy()
            out[f"m{idx}_{nm}_scales"] = mod.scales.float().numpy()
            out[f"m{idx}_{nm}_szeros"] = mod.scaled_zeros.float().numpy()
        for tokens in (1, 3, 7, 8, 9, 33):
            x = (torch.randn(tokens, K, generator=g) * 0.5).half()
            del calls[:]
            c = mlp.our_llama_mlp(x)
            assert len(calls) == 2 and {cc[0] for cc in calls} == ({"gemv"} if tokens < 8 else {"gemm"})
            out[f"m{idx}_t{tokens}_x"] = x.float().numpy()
            out[f"m{idx}_t{tokens}_c"] = c.float().numpy()
            if tokens >= 8:   # the zeros tensors the reference handed to the engine (fp16 arithmetic, :69,76)
                out[f"m{idx}_t{tokens}_gate_zeros_passed"] = calls[0][1].float().numpy()
                out[f"m{idx}_t{tokens}_up_zeros_passed"] = calls[1][1].float().numpy()
    np.savez_compressed(os.path.join(HERE, "reference_mlp_callsite.npz"), **out)
    print("wrote reference_mlp_callsite.npz", len(out), "arrays")


def callsites_golden():
    """tests/golden/reference_callsites.npz: the reference's own, unmodified call sites EXECUTED on CPU over a stub
    ``awq_inference_engine`` whose linears are the W4A16 oracle rounded to the element type, on the inputs of
    tests/test_reference_callsites_gpu.py (regenerated there from the same seeds):
      * awq.quantize.qmodule.WQLinear                the state dict of a 256 -> 64 layer; forward (qmodule.py:201-224):
                                                     which entry it calls, the bias added to the rounded output
      * tinychat.modules.fused_mlp.QuantLlamaMLP     our_llama_mlp (fused_mlp.py:36-83), both branches
      * tinychat.modules.fused_attn.make_quant_attn  the fused QKV WQLinear it builds (fused_attn.py:566-594): shapes and
                                                     sums of its buffers, and its outputs
    Outputs are stored at up to 4 seeded rows (callsite_rows) and every other column, as bit patterns of the element
    type."""
    root = os.path.dirname(os.path.dirname(HERE))
    for p in (root, os.path.join(root, "tests"), REF):
        if p not in sys.path:
            sys.path.insert(0, p)
    from oracle import w4a16_oracle as O
    from awq_testutil import gen_layer, gen_x
    from test_reference_callsites_gpu import MLP_TOKENS, QKV_TOKENS, WQ_SHAPES, callsite_rows, layer_bias
    # the one stub every reference module imported in this process holds: generators that ran before bound their own
    # entries onto it, so this one rebinds them rather than registering a second stub those modules would not see
    eng = sys.modules.setdefault("awq_inference_engine", types.ModuleType("awq_inference_engine"))
    calls = []

    def linear(x, qw, s, z):
        tag = "f16" if x.dtype == torch.float16 else "bf16"
        x2 = x.reshape(-1, x.shape[-1]).double().numpy()
        y = O.wq_linear_forward(x2, qw.numpy(), s.double().numpy(), z.double().numpy(), dtype=tag)
        return torch.from_numpy(O.rounder(tag)(y)).to(x.dtype).reshape(*x.shape[:-1], -1)

    def gemv(x, qw, s, z, m, n, k, g):
        calls.append("gemv")
        return linear(x, qw, s, z)

    def gemm(x, qw, s, z):
        calls.append("gemm")
        return linear(x, qw, s, z)
    eng.gemv_forward_cuda_new, eng.gemm_forward_cuda_new = gemv, gemm
    import contextlib
    with contextlib.redirect_stdout(sys.stderr):
        import awq.quantize.qmodule as qmodule
        import tinychat.utils.constants as constants
        constants.init()
        import tinychat.modules.fused_mlp as fused_mlp
        import tinychat.modules.fused_attn as fused_attn

    def ref_wqlinear(K, N, dtype, seed, bias=False):
        m = qmodule.WQLinear(4, 128, K, N, bias, "cpu", dtype=dtype)
        m.qweight, m.scales, m.scaled_zeros = gen_layer(N, K, dtype, seed=seed)
        if bias:
            m.bias = layer_bias(N, dtype, seed)
        return m
    bits = lambda t, M: t.reshape(M, -1)[callsite_rows(M)][:, ::2].contiguous().view(torch.int16).numpy()
    out = {}
    for k, v in qmodule.WQLinear(4, 128, 256, 64, False, "cpu").state_dict().items():   # the module's buffers
        out[f"state_{k}_shape"], out[f"state_{k}_dtype"] = np.array(v.shape), np.array(str(v.dtype))
    K, N = 1024, 768
    for tag, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
        for bias in (False, True):
            m = ref_wqlinear(K, N, dt, 5, bias)
            for shape in WQ_SHAPES:
                M = shape[0] * shape[1]
                x = gen_x(M, K, dt, seed=shape[1]).view(*shape, K)
                del calls[:]
                y = m(x)
                key = f"wq_{tag}_b{int(bias)}_{shape[0]}x{shape[1]}"
                out[key + "_y"] = bits(y, M)
                out[key + "_calls"] = np.array(calls)
    dt, H, I = torch.float16, 1024, 2816
    gate, up, down = ref_wqlinear(H, I, dt, 11), ref_wqlinear(H, I, dt, 12), ref_wqlinear(I, H, dt, 13)
    mlp = fused_mlp.QuantLlamaMLP(gate, down, up)
    for tokens in MLP_TOKENS:
        x = (gen_x(tokens, H, dt, seed=tokens) * 0.5).view(1, tokens, H)
        del calls[:]
        c = mlp.our_llama_mlp(x)
        out[f"mlp_t{tokens}_c"] = bits(c, tokens)
        out[f"mlp_t{tokens}_calls"] = np.array(calls)
    H, KV = 1024, 256

    class LlamaAttentionFused(torch.nn.Module):   # the class NAME is what make_quant_attn matches (:559-563)
        def __init__(self):
            super().__init__()
            self.q_proj, self.k_proj = ref_wqlinear(H, H, dt, 21), ref_wqlinear(H, KV, dt, 22)
            self.v_proj, self.o_proj = ref_wqlinear(H, KV, dt, 23), ref_wqlinear(H, H, dt, 24)
            self.args = types.SimpleNamespace(hidden_size=H, num_attention_heads=8, num_key_value_heads=2,
                                              max_position_embeddings=128, rope_theta=10000.0, rope_scaling=None)
            self.kv_max_seq_len = 64

    class Holder(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.attn = LlamaAttentionFused()
    model = Holder()
    with contextlib.redirect_stdout(sys.stderr):
        fused_attn.make_quant_attn(model, "cpu")
    qkv = model.attn.qkv_proj
    for nm in ("qweight", "scales", "scaled_zeros"):
        t = getattr(qkv, nm)
        out[f"qkv_{nm}_shape"] = np.array(t.shape)
        out[f"qkv_{nm}_sum"] = t.float().numpy().astype(np.float64).sum() if t.is_floating_point() else t.numpy().astype(np.int64).sum()
    for tokens in QKV_TOKENS:
        x = gen_x(tokens, H, dt, seed=30 + tokens).view(1, tokens, H)
        del calls[:]
        y = qkv(x)
        out[f"qkv_t{tokens}_y"] = bits(y, tokens)
        out[f"qkv_t{tokens}_calls"] = np.array(calls)
    np.savez_compressed(os.path.join(HERE, "reference_callsites.npz"), **out)
    print("wrote reference_callsites.npz", len(out), "arrays")


def kernels_golden(out_dir=HERE):
    """tests/golden/reference_kernels.npz: what the reference's own CUDA kernels, rebuilt for sm_100a by
    oracle/build_ref.py, return on the inputs of the GPU tests that compare against them.  Needs a CUDA device and
    oracle/_ref (run it where both exist):

        python tests/golden/make_golden.py --kernels [OUT_DIR]

    Stored (samples keep the file small; the tests regenerate the inputs from the same seeds):
      * W4A16 GEMV / GEMM (tests/test_gpu_parity.py::test_matches_reference_kernels): bit patterns of y at up to 16
        seeded rows and at the output columns 0, 74, 148, ..., plus the sums of x and qweight that identify the inputs
      * layernorm_forward_cuda (tests/test_layer_ops_gpu.py): bit patterns of 8192 seeded elements of the output
      * rotary_embedding_neox (tests/test_zz_rope_neox_gpu.py): bit patterns of 64 seeded (token, head) rows of q
        and of k after the in-place rotation"""
    root = os.path.dirname(os.path.dirname(HERE))
    for p in (root, os.path.join(root, "tests"), os.path.join(root, "oracle", "_ref")):
        if p not in sys.path:
            sys.path.insert(0, p)
    import ref_awq_engine as ref
    from awq_testutil import gen_layer, gen_x
    from test_gpu_parity import REF_KERNEL_CASES, ref_kernel_rows
    from test_layer_ops_gpu import rmsnorm_ref_inputs
    from test_zz_rope_neox_gpu import rope_ref_inputs
    dev = "cuda:0"
    out = {}
    for M, N, K in REF_KERNEL_CASES:
        for tag, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
            qw, s, z = gen_layer(N, K, dt, seed=9, device=dev)
            x = (gen_x(M, K, dt, seed=10, device=dev) * 0.25).contiguous()
            if M < 8:
                y = ref.gemv_forward_cuda_new(x, qw, s, z, M, N, K, 128)
            else:
                y = ref.gemm_forward_cuda_new(x, qw, s, z)
            torch.cuda.synchronize()
            key = f"w4_{M}x{N}x{K}_{tag}"
            out[key + "_y"] = y.cpu()[ref_kernel_rows(M)][:, ::74].contiguous().view(torch.int16).numpy()
            out[key + "_xsum"] = np.float64(x.float().cpu().numpy().astype(np.float64).sum())
            out[key + "_qwsum"] = np.int64(qw.cpu().numpy().astype(np.int64).sum())
    pick = np.random.default_rng(7)
    for tag, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
        x, gamma = rmsnorm_ref_inputs(dt, dev)
        y = torch.empty_like(x)
        ref.layernorm_forward_cuda(x, gamma, y, 1e-6)
        torch.cuda.synchronize()
        idx = np.sort(pick.choice(y.numel(), 32768, replace=False))[::4].astype(np.int32)
        out[f"rms_{tag}_idx"] = idx
        out[f"rms_{tag}_y"] = y.view(torch.int16).cpu().reshape(-1).numpy()[idx]
        pos, q, k, cache = rope_ref_inputs(dt, dev)
        ref.rotary_embedding_neox(pos, q, k, q.shape[-1], cache)
        torch.cuda.synchronize()
        for nm, t in (("q", q), ("k", k)):
            rows = t.reshape(-1, t.shape[-1])
            idx = np.sort(pick.choice(rows.shape[0], 256, replace=False))[::4].astype(np.int32)
            out[f"rope_{tag}_{nm}_idx"] = idx
            out[f"rope_{tag}_{nm}"] = rows.view(torch.int16).cpu().numpy()[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.savez_compressed(os.path.join(out_dir, "reference_kernels.npz"), **out)
    print("wrote reference_kernels.npz", len(out), "arrays")


def main():
    qmodule, pseudo_quantize_tensor = _import_reference()
    g = torch.Generator().manual_seed(20260922)
    out = {}

    # 1. pack_intweight on random nibbles, several shapes (incl. 11008-style non-pow2 K)
    for idx, (N, K) in enumerate([(4, 64), (8, 128), (16, 256), (32, 192), (64, 512), (128, 1024)]):
        q = torch.randint(0, 16, (N, K), generator=g, dtype=torch.int32)
        packed = qmodule.pack_intweight(q, interleave=4, kstride=64)
        out[f"pack{idx}_q"] = q.numpy().astype(np.uint8)
        out[f"pack{idx}_packed"] = packed.numpy()

    # 2. calculate_zeros_width table
    ins = [64, 128, 256, 1024, 3584, 4096, 5120, 8192, 11008, 14336, 28672]
    out["zw_in"] = np.array(ins)
    out["zw_g128"] = np.array([qmodule.calculate_zeros_width(i, 128) for i in ins])
    out["zw_g64"] = np.array([qmodule.calculate_zeros_width(i, 64) for i in ins])

    # 3. pseudo_quantize_tensor + WQLinear.from_linear, fp32 / fp16 / bf16 layers
    for tag, dt in (("f32", torch.float32), ("f16", torch.float16), ("bf16", torch.bfloat16)):
        N, K, G = 32, 256, 128
        lin = torch.nn.Linear(K, N, bias=True)
        with torch.no_grad():
            lin.weight.copy_(torch.randn(N, K, generator=g) * 0.02)
            lin.bias.copy_(torch.randn(N, generator=g) * 0.1)
        lin = lin.to(dt)
        w0 = lin.weight.data.clone()
        w_dq, scales, zeros = pseudo_quantize_tensor(
            lin.weight.data.clone(), n_bit=4, zero_point=True, q_group_size=G, get_scale_zp=True)
        lin.weight.data = w_dq            # real_quantize_model_weight does the same (quantizer.py:150-152)
        wq = qmodule.WQLinear.from_linear(lin, 4, G, False, scales, zeros)
        f = lambda t: t.detach().float().numpy()
        out[f"fl_{tag}_w0"] = f(w0)
        out[f"fl_{tag}_wdq"] = f(w_dq)
        out[f"fl_{tag}_scales"] = f(scales)
        out[f"fl_{tag}_zeros"] = f(zeros)
        out[f"fl_{tag}_qweight"] = wq.qweight.numpy()
        out[f"fl_{tag}_sbuf"] = f(wq.scales)
        out[f"fl_{tag}_zbuf"] = f(wq.scaled_zeros)
        out[f"fl_{tag}_bias"] = f(wq.bias)
        assert tuple(wq.qweight.shape) == (N // 4, K) and wq.qweight.dtype == torch.int16

    # 3b. out-of-range integers through pack_intweight (unmasked OR, qmodule.py:50-55) and from_linear on
    #     RAW (not fake-quantised) weights, where round((w + s*z)/s) can leave 0..15 in half precision
    q = torch.randint(-3, 19, (16, 128), generator=g, dtype=torch.int32)
    out["packoob_q"] = q.numpy().astype(np.int32)
    out["packoob_packed"] = qmodule.pack_intweight(q, interleave=4, kstride=64).numpy()
    for tag, dt in (("f16", torch.float16), ("bf16", torch.bfloat16)):
        N, K, G = 32, 256, 128
        lin = torch.nn.Linear(K, N, bias=False)
        with torch.no_grad():
            lin.weight.copy_(torch.randn(N, K, generator=g) * 0.02)
        lin = lin.to(dt)
        _, scales, zeros = pseudo_quantize_tensor(
            lin.weight.data.clone(), n_bit=4, zero_point=True, q_group_size=G, get_scale_zp=True)
        wq = qmodule.WQLinear.from_linear(lin, 4, G, False, scales, zeros)
        f = lambda t: t.detach().float().numpy()
        out[f"flraw_{tag}_w"] = f(lin.weight.data)
        out[f"flraw_{tag}_scales"] = f(scales)
        out[f"flraw_{tag}_zeros"] = f(zeros)
        out[f"flraw_{tag}_qweight"] = wq.qweight.numpy()
        out[f"flraw_{tag}_sbuf"] = f(wq.scales)
        out[f"flraw_{tag}_zbuf"] = f(wq.scaled_zeros)

    # 4. buffer shapes declared by WQLinear.__init__ for the BASELINE shapes
    shapes = []
    for (K, N) in [(4096, 4096), (4096, 6144), (4096, 14336), (14336, 4096), (8192, 1280),
                   (1024, 8192), (8192, 3584), (3584, 8192), (11008, 4096)]:
        m = qmodule.WQLinear(4, 128, K, N, False, "cpu")
        shapes.append([K, N, *m.qweight.shape, *m.scales.shape, *m.scaled_zeros.shape])
    out["init_shapes"] = np.array(shapes)

    np.savez_compressed(os.path.join(HERE, "reference_packer.npz"), **out)
    print("wrote", os.path.join(HERE, "reference_packer.npz"), len(out), "arrays")


if __name__ == "__main__":
    if "--kernels" in sys.argv:
        rest = sys.argv[sys.argv.index("--kernels") + 1:]
        kernels_golden(rest[0] if rest else HERE)
    else:
        main()
        repacker_golden()
        layer_ops_golden()
        mlp_callsite_golden()
        callsites_golden()
