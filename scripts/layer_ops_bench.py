#!/usr/bin/env python
"""Timing of the ops around the linears (SURVEY.md §8f) against their HBM bounds: RMSNorm, the one-kernel MLP front half,
decode attention.  CUDA graph of the plugin / C-ABI calls over buffers larger than L2 where the op streams data.
    python scripts/layer_ops_bench.py > gpurun_out/layer_ops.json"""
import ctypes
import json
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import llm_awq_b200 as P  # noqa: E402
from bench import read_peaks, alg_bytes, scale_rows  # noqa: E402

dev = torch.device("cuda", 0)
eng, lib, peaks = P.engine(), P.lib(), read_peaks()
out = {}


def timed(fn, iters=20):
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        fn()
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    for _ in range(3):
        g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters * 1e3   # us per graph replay


# ---- RMSNorm: 2 * m * n * 2 bytes
for m, n in ((2048, 4096), (1, 4096), (2048, 8192)):
    reps = max(1, (512 << 20) // (m * n * 4))
    xs = [torch.randn(m, n, device=dev).half() for _ in range(reps)]
    ys = [torch.empty_like(x) for x in xs]
    gamma = torch.ones(n, device=dev).half()
    us = timed(lambda: [eng.layernorm_forward_cuda(x.view(1, m, n), gamma, y.view(1, m, n), 1e-5) for x, y in zip(xs, ys)]) / reps
    b = 2 * m * n * 2
    out["rmsnorm_%dx%d" % (m, n)] = {"us": round(us, 3), "GBs": round(b / us / 1e3, 1), "hbm_frac": round(b / us / 1e3 / peaks["hbm"], 3)}

# ---- MLP front half, one token, Llama-3-8B: 2 weight sets of 14336 x 4096
N, K = 14336, 4096
reps = 12
layers = []
for i in range(reps):
    t = []
    for j in range(2):
        qw = torch.randint(-32768, 32768, (N // 4, K), dtype=torch.int32, device=dev).to(torch.int16)
        sc = (0.004 + 0.012 * torch.rand(scale_rows(K), N, device=dev)).half()
        sz = (-(sc.float() * torch.randint(0, 16, (scale_rows(K), N), device=dev))).half()
        t += [qw, sc, sz]
    layers.append(t)
x = (torch.randn(1, K, device=dev) * 0.25).half()
us_f = timed(lambda: [eng.mlp_front_forward_cuda(x, *t) for t in layers]) / reps
us_2 = timed(lambda: [torch.nn.functional.silu(eng.gemv_forward_cuda_new(x, *t[:3], 1, N, K, 128)) *
                      eng.gemv_forward_cuda_new(x, *t[3:], 1, N, K, 128) for t in layers]) / reps
b = 2 * alg_bytes(1, N, K) - 2 * K
out["mlp_front_one_token_14336x4096"] = {"us_one_kernel": round(us_f, 3), "us_reference_composition_on_this_plugin": round(us_2, 3),
                                         "hbm_frac_one_kernel": round(b / us_f / 1e3 / peaks["hbm"], 3)}

# ---- decode attention, Llama-3-8B heads (32 q, 8 kv, d 128), batch 1
H, Hkv, D = 32, 8, 128
for L, t in ((2048, 2047), (8192, 8191)):
    layers_n = 32
    kcs = [torch.randn(1, Hkv, D // 8, L, 8, device=dev).half() for _ in range(layers_n)]
    vcs = [torch.randn(1, Hkv, L, D, device=dev).half() for _ in range(layers_n)]
    q = torch.randn(1, H, D, device=dev).half()
    k = torch.randn(1, Hkv, D, device=dev).half()
    v = torch.randn(1, Hkv, D, device=dev).half()
    us = timed(lambda: [eng.single_query_attention(q, k, v, kc, vc, None, None, t, D, 500000.0, 1.0, True) for kc, vc in zip(kcs, vcs)]) / layers_n
    b = 2 * (t + 1) * D * 2 * Hkv
    out["attention_ctx%d" % (t + 1)] = {"us": round(us, 3), "GBs": round(b / us / 1e3, 1), "hbm_frac": round(b / us / 1e3 / peaks["hbm"], 3),
                                        "kv_bytes": b}

# ---- decode attention at other query-to-KV head ratios G = H / Hkv: the CUDA-core kernel (G <= 8) and the tensor-core
# kernel (G > 8).  Enough caches per graph to stream >= 384 MB (3x L2) per replay; one launch per cache.
for name, H, Hkv, D, batches in (("qwen2_7b", 28, 4, 128, (1,)), ("qwen2_1p5b", 12, 2, 128, (1,)),
                                  ("g16", 128, 8, 64, (1, 8)), ("mqa71", 71, 1, 64, (1, 8))):
    G = H // Hkv
    for B in batches:
        for L in (2048, 8192):
            t = L - 1
            b = 2 * B * (t + 1) * D * 2 * Hkv
            n = max(4, min(512, -(-(384 << 20) // b)))
            kcs = [torch.randn(B, Hkv, D // 8, L, 8, device=dev).half() for _ in range(n)]
            vcs = [torch.randn(B, Hkv, L, D, device=dev).half() for _ in range(n)]
            q = torch.randn(B, H, D, device=dev).half()
            k = torch.randn(B, Hkv, D, device=dev).half()
            v = torch.randn(B, Hkv, D, device=dev).half()
            us = timed(lambda: [eng.single_query_attention(q, k, v, kc, vc, None, None, t, D, 1000000.0, 1.0, True)
                                for kc, vc in zip(kcs, vcs)]) / n
            row = {"G": G, "kernel": "tensor_core" if G > 8 else "cuda_core", "us": round(us, 3), "kv_bytes": b,
                   "GBs": round(b / us / 1e3, 1), "hbm_frac": round(b / us / 1e3 / peaks["hbm"], 3), "caches_per_replay": n}
            if G > 8:
                flop = 4 * B * H * (t + 1) * D
                t_hbm, t_tc = b / (peaks["hbm"] * 1e3), flop / (peaks["tc_burst"] * 1e6)   # us
                row.update({"flop": flop, "TFLOPs": round(flop / us / 1e6, 2), "bound": "hbm" if t_hbm >= t_tc else "tensor",
                            "hbm_bound_us": round(t_hbm, 3), "tc_bound_us": round(t_tc, 3)})
            out["attention_%s_b%d_ctx%d" % (name, B, L)] = row
            del kcs, vcs
out["peaks"] = dict(peaks)
try:
    import subprocess
    out["device"] = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                   capture_output=True, text=True).stdout.strip()
except OSError:
    out["device"] = torch.cuda.get_device_name(0)
print(json.dumps(out, indent=1))
