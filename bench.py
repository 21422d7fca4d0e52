#!/usr/bin/env python
"""Benchmark of the W4A16 linear path (BASELINE.json metric): Llama-3-8B W4A16 g128, 1 x B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference|reference-gpu]

A "step" is ONE pass of the hot path over one batch of synthetic input:
  decode  (headline, BASELINE configs[1]): the 160 W4A16 GEMVs of one token, 32 layers x
          {qkv 4096->6144, o 4096->4096, gate/up 4096->14336, down 14336->4096}, M = 1, all 32
          layers' weights distinct (3.7 GB >> the 126 MB L2, so every weight byte is an HBM read;
          that is the "inputs larger than L2" timing rule), executed in model order.
  prefill (BASELINE configs[2], reported in the same line under "prefill"): the same 160 layers
          with M = 2048 tokens through the tcgen05 tensor-core kernel.
`value`  = tokens/s of the linear path with inputs resident in HBM: the 160 launches of a step are a
           CUDA graph of C-ABI launches (include/b200awq.h), K steps timed with CUDA events.
`e2e`    = the same metric through the reference-facing plugin (`awq_inference_engine.
           gemv_forward_cuda_new` / `gemm_forward_cuda_new`, the calls WQLinear.forward makes) with
           HOST buffers: every step copies the step's activations from pinned host memory, runs the
           160 plugin calls and copies the result back; the host waits for the result every step.
Synthetic data: random int16 packed weights (every bit pattern is a legal packing), scales
0.004..0.016, integer zero points, N(0,1) activations (SURVEY.md §8d).  Multi-GPU: the model fits
one GPU, so N ranks are N independent replicas (no data-path collective; "scaling": "weak").
"""
import argparse
import ctypes
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

LLAMA3_8B = dict(name="Llama-3-8B", hidden=4096, inter=14336, q_heads=32, kv_heads=8, head_dim=128, layers=32)
LLAMA2_70B = dict(name="Llama-2-70B", hidden=8192, inter=28672, q_heads=64, kv_heads=8, head_dim=128, layers=80)
METRIC = "Llama-3-8B W4A16 g128 decode tok/s (linear path), %dxB200"
UNIT = "tok/s"
G = 128


def layer_projs(cfg):
    """(name, K, N) of the five quantised linears of one decoder layer after tinychat's QKV fusion
    (tinychat/modules/fused_attn.py:566-594), in execution order."""
    h, it, hd = cfg["hidden"], cfg["inter"], cfg["head_dim"]
    return [("qkv", h, (cfg["q_heads"] + 2 * cfg["kv_heads"]) * hd), ("o", cfg["q_heads"] * hd, h),
            ("gate", h, it), ("up", h, it), ("down", it, h)]


def alg_bytes(M, N, K):
    """Algorithmic bytes of one call: qweight + scales + scaled_zeros (unpadded rows) + x + y."""
    return N * K // 2 + 2 * (K // G) * N * 2 + 2 * M * K + 2 * M * N


def alg_flops(M, N, K):
    return 2 * M * N * K


def scale_rows(K):
    return ((K // G + 7) // 8) * 8


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tc_burst=d["bf16_tflops"], tc_sustained=d["bf16_tflops_sustained"], source="measured")
    return dict(hbm=6650.0, tc_burst=1590.0, tc_sustained=1400.0, source="fallback")


# ------------------------------------------------------------------------------------------ clocks
class ClockSampler:
    """Samples SM clock / throttle reasons with NVML on a background thread during the timed regions."""

    def __init__(self, index):
        self.samples, self.stop_flag, self.thread, self.ok = [], False, None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:  # noqa: BLE001
            self.err = repr(e)

    def _run(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:  # noqa: BLE001
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.samples.append((time.time(), mhz, reasons, util))
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.02)

    def start(self):
        if self.ok:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def stop(self, windows):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.stop_flag = True
        self.thread.join()
        inside = [s for s in self.samples if any(a <= s[0] <= b for a, b in windows)] or self.samples
        names = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown",
                 0x10: "sync_boost", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
                 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}
        seen = set()
        for s in inside:
            for bit, nm in names.items():
                if s[2] & bit and nm != "gpu_idle":
                    seen.add(nm)
        return {"sm_mhz": statistics.median([s[1] for s in inside]) if inside else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(seen), "samples": len(inside)}


# ------------------------------------------------------------------------------------------ model
def tp_projs(cfg, tp):
    """Per-rank shapes under tensor parallelism (SURVEY.md §8e): qkv / gate / up column-parallel
    (N / tp), o / down row-parallel (K / tp, followed by ONE all-reduce)."""
    out = []
    for name, K, N in layer_projs(cfg):
        if name in ("o", "down"):
            out.append((name, K // tp, N))
        else:
            out.append((name, K, N // tp))
    return out


def build_model(torch, cfg, dtype, device, layers=None, projs=None):
    """Packed weights of every quantised linear, generated on the device (SURVEY.md §8d generator)."""
    out = []
    for l in range(cfg["layers"] if layers is None else layers):
        for p, (name, K, N) in enumerate(projs or layer_projs(cfg)):
            g = torch.Generator(device=device).manual_seed(1234 + 97 * l + p)
            qw = torch.randint(-32768, 32768, (N // 4, K), generator=g, dtype=torch.int32, device=device).to(torch.int16)
            rows, ng = scale_rows(K), K // G
            sc = torch.zeros(rows, N, device=device)
            sc[:ng] = 0.004 + 0.012 * torch.rand(ng, N, generator=g, device=device)
            sc = sc.to(dtype)
            zi = torch.randint(0, 16, (rows, N), generator=g, device=device)
            sz = (-(sc.float() * zi)).to(dtype)
            sz[ng:] = 0
            out.append(dict(name=name, K=K, N=N, qw=qw, sc=sc, sz=sz))
    return out


def dist_setup(torch, n_gpus):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        return rank, world, local, dist
    torch.cuda.set_device(local)
    return rank, world, local, None


def max_over_ranks(torch, dist, ms, device):
    if dist is None:
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(torch, dist):
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()


def timed_steps(torch, dist, device, step_fn, steps, warmup, sync_each=False):
    """W untimed + exactly K timed steps, barrier + synchronize on both sides, CUDA events on the
    launching stream, max over ranks.  Returns (ms_total, (t0, t1) wall window)."""
    for _ in range(warmup):
        step_fn()
        if sync_each:
            torch.cuda.current_stream().synchronize()
    barrier(torch, dist)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    for _ in range(steps):
        step_fn()
        if sync_each:
            torch.cuda.current_stream().synchronize()
    e1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    ms = e0.elapsed_time(e1)
    barrier(torch, dist)
    return max_over_ranks(torch, dist, ms, device), (t0, t1)


# ------------------------------------------------------------------------------------------ arms
def run_b200(args):
    import torch
    import llm_awq_b200 as P
    rank, world, local, dist = dist_setup(torch, args.gpus)
    device = torch.device("cuda", local)
    dtype = torch.float16
    lib, eng = P.lib(), P.engine()
    cfg = LLAMA3_8B
    peaks = read_peaks()
    sampler = ClockSampler(local)
    model = build_model(torch, cfg, dtype, device)
    nl = len(model)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    windows = []

    def make_inputs(M, scale=1.0):
        g = torch.Generator(device=device).manual_seed(99 + M)
        return {K: (torch.randn(M, K, generator=g, device=device) * scale).to(dtype) for K in (cfg["hidden"], cfg["inter"])}

    def abi_graph(M, kind, per_layer=False):
        """CUDA graph of one step: 160 launches through the C ABI on the capture stream.  Outputs: one buffer per
        layer with `per_layer`, else one per output width (each layer overwrites the previous one's)."""
        xs = make_inputs(M)
        ys = {N: torch.empty(M, N, dtype=dtype, device=device) for N in {m["N"] for m in model}}
        outs = [torch.empty(M, m["N"], dtype=dtype, device=device) for m in model] if per_layer else [ys[m["N"]] for m in model]
        fn = lib.b200awq_w4a16_gemv if kind == "gemv" else lib.b200awq_w4a16_gemm

        def launch_all():
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            for m, y in zip(model, outs):
                a = (p(xs[m["K"]]), p(m["qw"]), p(m["sc"]), p(m["sz"]), p(y), M, m["N"], m["K"], G, 0)
                rc = fn(*a, st) if kind == "gemv" else fn(*a, None, 0, st)
                if rc != 0:
                    raise RuntimeError(lib.b200awq_strerror(rc).decode())
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            launch_all()
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            launch_all()
        return g, (xs, outs)

    def plugin_graph(M, kind):
        """CUDA graph of one e2e step: H2D of the activations (pinned), 160 plugin calls, D2H of the result."""
        hx = {K: v.cpu().pin_memory() for K, v in make_inputs(M).items()}
        dx = {K: torch.empty_like(v, device=device) for K, v in hx.items()}
        hy = torch.empty(M, cfg["hidden"], dtype=dtype).pin_memory()

        def run():
            for K in dx:
                dx[K].copy_(hx[K], non_blocking=True)
            y = None
            for m in model:
                x = dx[m["K"]]
                if kind == "gemv":
                    y = eng.gemv_forward_cuda_new(x, m["qw"], m["sc"], m["sz"], M, m["N"], m["K"], G)
                else:
                    y = eng.gemm_forward_cuda_new(x, m["qw"], m["sc"], m["sz"])
            hy.copy_(y, non_blocking=True)
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            run()
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            run()
        h2d = sum(v.numel() * 2 for v in hx.values())
        return g, hy, h2d, hy.numel() * 2

    def eager_e2e(M, steps):
        """The SAME end-to-end step without a CUDA graph: every layer is one eager call of the reference-facing module
        (this repo's mirror of WQLinear.forward), as tinychat / awq.entry make them; pinned H2D of the activations and
        D2H of the result every step."""
        mods, kind = reference_wqlinears(torch, model, device, dtype)
        hx = {K: v.cpu().pin_memory() for K, v in make_inputs(M).items()}
        dx = {K: torch.empty_like(v, device=device).view(1, M, K) for K, v in hx.items()}
        hy = torch.empty(1, M, cfg["hidden"], dtype=dtype).pin_memory()

        def step():
            for K in dx:
                dx[K].copy_(hx[K].view(1, M, K), non_blocking=True)
            y = None
            for m, mod in zip(model, mods):
                y = mod(dx[m["K"]])
            hy.copy_(y, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            _ = float(hy[0, 0, 0])
        ms, w = timed_steps(torch, dist, device, step, steps, args.warmup)
        # host cost of one call when the GPU is not the bottleneck: issue the calls of one step and stop the clock before
        # waiting for the device
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for m, mod in zip(model, mods):
            mod(dx[m["K"]])
        host_us = (time.perf_counter() - t0) * 1e6 / nl
        torch.cuda.synchronize()
        return ms / steps, host_us, kind, w

    def batch_sweep():
        """BASELINE configs[4]: the five Llama-3-8B shapes at M in {1, 4, 16, 64} through the C ABI (the reference
        dispatch: GEMV entry below 8 tokens, GEMM entry from 8), each shape over its 32 distinct layers (> L2), CUDA
        graph + events.  us per call and fraction of the HBM roofline (the whole sweep is HBM-bound, SURVEY.md §8d)."""
        out = {}
        shapes = sorted({(m["N"], m["K"]) for m in model})
        for M in (1, 4, 16, 64):
            xs = make_inputs(M)
            row = {}
            for (N, K) in shapes:
                layers = [m for m in model if (m["N"], m["K"]) == (N, K)]
                y = torch.empty(M, N, dtype=dtype, device=device)

                def launch_all():
                    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
                    for m in layers:
                        a = (p(xs[K]), p(m["qw"]), p(m["sc"]), p(m["sz"]), p(y), M, N, K, G, 0)
                        rc = lib.b200awq_w4a16_gemv(*a, st) if M < 8 else lib.b200awq_w4a16_gemm(*a, None, 0, st)
                        if rc != 0:
                            raise RuntimeError(lib.b200awq_strerror(rc).decode())
                s = torch.cuda.Stream()
                with torch.cuda.stream(s):
                    launch_all()
                s.synchronize()
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    launch_all()
                ms, _ = timed_steps(torch, None, device, g.replay, args.steps, args.warmup)
                us = ms * 1e3 / args.steps / len(layers)
                row["%dx%d" % (N, K)] = {"us": round(us, 3), "frac": round(alg_bytes(M, N, K) / us / 1e3 / peaks["hbm"], 4),
                                         "calls": len(layers)}
            tot_us = sum(v["us"] * v["calls"] for v in row.values())
            row["tok_s"] = round(M * 1e6 / tot_us, 1)
            row["frac"] = round(sum(alg_bytes(M, m["N"], m["K"]) for m in model) / tot_us / 1e3 / peaks["hbm"], 4)
            out[str(M)] = row
        return out

    # outputs of the last timed step of each leg (--dump-outputs); prefill outputs at fixed seeded rows
    dump = {}
    rows_p = torch.from_numpy(np.sort(np.random.default_rng(0).choice(2048, 64, replace=False)))

    def keep(name, t):
        dump[name] = t.float().cpu().numpy()

    sampler.start()
    # ---------------- decode: device-resident
    g_dec, keep1 = abi_graph(1, "gemv", per_layer=True)
    ms_dec, w = timed_steps(torch, dist, device, g_dec.replay, args.steps, args.warmup)
    windows.append(w)
    for name, _, _ in layer_projs(cfg):
        keep("decode_" + name, torch.cat([y for m, y in zip(model, keep1[1]) if m["name"] == name]))
    # ---------------- decode: end to end through the plugin with host buffers
    g_e2e, hy, h2d, d2h = plugin_graph(1, "gemv")

    def e2e_step():
        g_e2e.replay()
        torch.cuda.current_stream().synchronize()
        _ = float(hy[0, 0])            # the host reads the step's result
    ms_e2e, w = timed_steps(torch, dist, device, e2e_step, args.steps, args.warmup)
    windows.append(w)
    keep("decode_e2e_y", hy)
    # ---------------- prefill (secondary object)
    Mp = 2048
    ksteps_p = args.steps if args.prefill_steps is None else args.prefill_steps
    g_pre, keep2 = abi_graph(Mp, "gemm")
    ms_pre, w = timed_steps(torch, dist, device, g_pre.replay, ksteps_p, args.warmup)
    windows.append(w)
    last = {m["N"]: (m["name"], y) for m, y in zip(model, keep2[1])}   # each buffer holds its last writer's output
    for name, y in last.values():
        keep(f"prefill_{name}_last_layer", y[rows_p.to(device)])
    g_pe2e, hyp, h2dp, d2hp = plugin_graph(Mp, "gemm")

    def pe2e_step():
        g_pe2e.replay()
        torch.cuda.current_stream().synchronize()
        _ = float(hyp[0, 0])
    ms_pe2e, w = timed_steps(torch, dist, device, pe2e_step, ksteps_p, args.warmup)
    windows.append(w)
    keep("prefill_e2e_y", hyp[rows_p])
    keep("prefill_rows", rows_p)
    # ---------------- decode end to end WITHOUT a graph (what an unmodified caller sees)
    ms_eager, host_us, eager_kind, w = eager_e2e(1, args.steps)
    windows.append(w)
    sweep = batch_sweep() if (world == 1 and args.sweep) else None
    clocks = sampler.stop(windows)
    tp = None
    bytes_step = sum(alg_bytes(1, m["N"], m["K"]) for m in model)
    flops_step = sum(alg_flops(Mp, m["N"], m["K"]) for m in model)
    weights_bytes = sum(m["qw"].numel() * 2 for m in model)
    if world > 1:
        del g_dec, g_e2e, g_pre, g_pe2e, keep1, keep2
        model.clear()
        torch.cuda.empty_cache()
        tp = tp70b_measure(torch, dist, rank, world, device, args.steps, args.warmup)

    if rank != 0:
        return
    if args.dump_outputs:
        write_outputs(args.dump_outputs, dump)
    step_ms = ms_dec / args.steps
    ach = bytes_step / (step_ms * 1e-3) / 1e9
    traffic = None
    tf = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tf):
        traffic = json.load(open(tf)).get("decode_dram_bytes_per_launch")
    pre_ms = ms_pre / ksteps_p
    tfl = flops_step / (pre_ms * 1e-3) / 1e12
    line = {
        "metric": METRIC % world, "value": world * 1000.0 / step_ms, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": step_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16", "data": "synthetic",
        "config": {"workload": "Llama-3-8B W4A16 g128 decode bs=1: 32 layers x {qkv,o,gate,up,down} GEMV (BASELINE configs[1])",
                   "launches_per_step": nl, "weights_bytes": weights_bytes,
                   "l2": "inputs larger than L2 (3.7 GB of distinct weights per step, model order)",
                   "parallelism": "replicas x%d (model fits one GPU; no collective)" % world, "accumulate": "fp32"},
        "e2e": {"value": world * 1000.0 * args.steps / ms_e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps,
                "api": "awq_inference_engine.gemv_forward_cuda_new x160 in a CUDA graph with the pinned H2D/D2H copies; host sync + read every step"},
        "e2e_eager": {"value": world * 1000.0 / ms_eager, "unit": UNIT, "ms_per_step": ms_eager, "host_us_per_call": host_us,
                      "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                      "api": eager_kind + ".forward x160, eager launches (no CUDA graph), pinned H2D/D2H + host read every step"},
        "gpu_launches": nl * args.steps,
        "roofline": {"bound": "hbm", "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s", "frac": ach / peaks["hbm"],
                     "traffic": traffic, "kernel": "w4a16_decode_kernel", "peak_source": peaks["source"] + " (burst copy)",
                     "bytes_per_launch": bytes_step / nl, "avg_launch_us": step_ms * 1e3 / nl},
        "clocks": clocks,
        "prefill": {"metric": "Llama-3-8B W4A16 g128 prefill tok/s (linear path), seq=2048 (BASELINE configs[2])",
                    "value": world * Mp * 1000.0 / pre_ms, "unit": UNIT, "steps": ksteps_p, "ms_per_step": pre_ms,
                    "e2e": {"value": world * Mp * 1000.0 * ksteps_p / ms_pe2e, "unit": UNIT, "h2d_bytes_per_step": h2dp,
                            "d2h_bytes_per_step": d2hp},
                    "gpu_launches": nl * ksteps_p,
                    "roofline": {"bound": "tensor", "achieved": tfl, "peak": peaks["tc_sustained"], "unit": "TFLOP/s",
                                 "frac": tfl / peaks["tc_sustained"], "traffic": None, "kernel": "w4a16_umma_kernel",
                                 "peak_source": peaks["source"] + " (sustained cuBLAS bf16)", "frac_of_burst": tfl / peaks["tc_burst"]}},
    }
    if sweep is not None:
        line["batch_sweep"] = sweep
    if tp is not None:
        line["tp70b"] = tp
    ptf = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(ptf):
        line["prefill"]["roofline"]["traffic"] = json.load(open(ptf)).get("prefill_dram_bytes_per_launch")
    if world == 1 and not args.no_cpu:
        line["cpu_baseline"] = cpu_baseline(args.cpu_seconds)
    if world == 1 and args.ref_gpu:
        try:
            line["reference_on_b200"] = reference_gpu(torch, model, make_inputs, device, args.steps, lib)
        except Exception as e:  # noqa: BLE001
            line["reference_on_b200"] = {"unavailable": repr(e)[:200]}
    print(json.dumps(line))


def write_outputs(out_dir, arrays):
    """DIR/<name>.npy, float32, for comparing two builds output for output (the inputs are seeded)."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float32))


def reference_wqlinears(torch, model, device, dtype):
    """One reference-facing module per layer of `model`, sharing the layer's packed buffers: this repo's mirror of the
    reference's WQLinear."""
    import llm_awq_b200 as P
    P.engine()
    mods = []
    for m in model:
        mod = P.WQLinear(4, G, 128, 8, False, "cpu")   # tiny buffers, replaced below
        mod.in_features, mod.out_features = m["K"], m["N"]
        mod.qweight, mod.scales, mod.scaled_zeros = m["qw"], m["sc"], m["sz"]
        mods.append(mod)
    return mods, "llm_awq_b200.WQLinear (mirror of the reference module)"


def tp70b_measure(torch, dist, rank, world, device, steps, warmup):
    """BASELINE configs[3]: Llama-2-70B W4A16 decode bs=1, tensor-parallel over the ranks of this launch.
    Per layer and rank: qkv (col) -> o (row, all-reduce) -> gate, up (col) -> down (row, all-reduce); the
    160 all-reduces of one token are 16 KB each (latency-bound).  Total work is fixed: "strong" scaling.
    Returns the record (rank 0) or None."""
    import llm_awq_b200 as P
    dtype = torch.float16
    lib = P.lib()
    cfg = LLAMA2_70B
    peaks = read_peaks()
    projs = tp_projs(cfg, world)
    model = build_model(torch, cfg, dtype, device, projs=projs)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    xs = {K: (torch.randn(1, K, device=device) * 0.25).to(dtype) for K in {m["K"] for m in model}}
    ys = {(m["name"], m["N"]): torch.empty(1, m["N"], dtype=dtype, device=device) for m in model}

    ex = None
    if world > 1:
        from llm_awq_b200 import tp
        ex = tp.PeerExchange(1, cfg["hidden"])

    def step(mode):
        """mode: "none" (no reduction, timing reference) | "nccl" (kernel + NCCL all-reduce) | "fused" (one kernel)"""
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        for m in model:
            y = ys[(m["name"], m["N"])]
            a = (p(xs[m["K"]]), p(m["qw"]), p(m["sc"]), p(m["sz"]), p(y), 1, m["N"], m["K"], G, 0)
            if mode == "fused" and m["name"] in ("o", "down"):
                rc = lib.b200awq_w4a16_gemv_allreduce(*a, ex.ptr, st)
            else:
                rc = lib.b200awq_w4a16_gemv(*a, st)
            if rc != 0:
                raise RuntimeError(lib.b200awq_strerror(rc).decode())
            if mode == "nccl" and dist is not None and m["name"] in ("o", "down"):
                dist.all_reduce(y)

    def graph(mode):
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            step(mode)
        s.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step(mode)
        return g
    ms_nc, _ = timed_steps(torch, dist, device, graph("none").replay, steps, warmup)
    ms_nccl = ms_fused = None
    if world > 1:
        ms_nccl, _ = timed_steps(torch, dist, device, graph("nccl").replay, steps, warmup)
        ms_fused, _ = timed_steps(torch, dist, device, graph("fused").replay, steps, warmup)
        # the exchange's watchdog poisons the outputs with NaN when a peer never delivered: such a timing is void
        bad = torch.tensor([0 if all(bool(torch.isfinite(y).all()) for y in ys.values()) else 1], device=device)
        dist.all_reduce(bad)
        if int(bad.item()):
            ms_fused = None
    ms_full = ms_nc if world == 1 else (ms_nccl if ms_fused is None else min(ms_nccl, ms_fused))
    if rank != 0:
        return None
    step_ms = ms_full / steps
    bytes_rank = sum(alg_bytes(1, m["N"], m["K"]) for m in model)
    return {
        "metric": "Llama-2-70B W4A16 g128 decode tok/s (linear path), TP=%d" % world, "value": 1000.0 / step_ms, "unit": UNIT,
        "n_gpus": world, "steps": steps, "warmup": warmup, "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
        "config": {"workload": "Llama-2-70B W4A16 g128 decode bs=1, TP=%d (BASELINE configs[3])" % world,
                   "parallelism": "tp%d: column-parallel qkv/gate/up, row-parallel o/down + 1 all-reduce each (NCCL, or fused into the GEMV over NVLink peer memory)" % world,
                   "launches_per_step": len(model), "allreduces_per_step": 0 if world == 1 else 2 * cfg["layers"],
                   "allreduce_bytes": cfg["hidden"] * 2, "l2": "inputs larger than L2"},
        "comm": {"ms_per_step_without_allreduce": ms_nc / steps,
                 "ms_per_step_nccl_allreduce": None if ms_nccl is None else ms_nccl / steps,
                 "ms_per_step_fused_nvlink_exchange": None if ms_fused is None else ms_fused / steps,
                 "headline_uses": "single GPU" if world == 1 else ("fused" if ms_fused is not None and ms_fused <= ms_nccl else "nccl")},
        "gpu_launches": len(model) * steps,
        "roofline": {"bound": "hbm", "achieved": bytes_rank / (step_ms * 1e-3) / 1e9, "peak": peaks["hbm"], "unit": "GB/s",
                     "frac": bytes_rank / (step_ms * 1e-3) / 1e9 / peaks["hbm"], "traffic": None, "per": "rank",
                     "frac_without_allreduce": bytes_rank / (ms_nc / steps * 1e-3) / 1e9 / peaks["hbm"]}}


def run_tp70b(args):
    import torch
    rank, world, local, dist = dist_setup(torch, args.gpus)
    rec = tp70b_measure(torch, dist, rank, world, torch.device("cuda", local), args.steps, args.warmup)
    if rec is not None:
        print(json.dumps(rec))


def cpu_layer(torch, layers=1):
    """One decoder layer's five WQLinear forwards (M = 1) on the host: the bounded CPU sample."""
    from oracle import cpu_path
    cfg = LLAMA3_8B
    model = build_model(torch, cfg, torch.float16, torch.device("cpu"), layers=layers)
    xs = {K: torch.randn(1, K).to(torch.float16) for K in (cfg["hidden"], cfg["inter"])}

    def step():
        y = None
        for m in model:
            y = cpu_path.wq_linear_forward(xs[m["K"]], m["qw"], m["sc"], m["sz"])
        return y
    return step


def pick_cpu_threads(torch, step):
    """All host threads is not always the fastest for these memory-bound elementwise ops (oversubscription):
    time one step with all cores, 32 and 16 threads and keep the best.  Returns the thread count used."""
    cores = os.cpu_count() or 1
    best, best_t = cores, None
    for n in sorted({cores, min(cores, 32), min(cores, 16)}, reverse=True):
        torch.set_num_threads(n)
        step()
        t0 = time.time()
        step()
        dt = time.time() - t0
        if best_t is None or dt < best_t:
            best, best_t = n, dt
    torch.set_num_threads(best)
    return best


def cpu_baseline(budget_s=15.0):
    """The pure-PyTorch dequant path (oracle/cpu_path.py) on the host cores: one decoder layer per
    sample step (1/32 of a token), repeated for about `budget_s` seconds."""
    import torch
    step = cpu_layer(torch)
    pick_cpu_threads(torch, step)
    ts, t_end = [], time.time() + budget_s
    while time.time() < t_end or len(ts) < 3:
        t0 = time.time()
        step()
        ts.append(time.time() - t0)
    med = statistics.median(ts)
    return {"value": 1.0 / (med * LLAMA3_8B["layers"]), "unit": UNIT, "cores": torch.get_num_threads(),
            "host_cores": os.cpu_count(), "kind": "port",
            "sample": "1 of 32 decoder layers (5 WQLinear forwards, M=1, dequant every call, fp32 torch ops), %d repeats, median; "
                      "tok/s = 1 / (32 x layer time)" % len(ts)}


def kernel_only_ms(torch, step):
    """Sum of the DEVICE durations of the kernels one step launches (CUPTI through torch.profiler): the time the GPU
    spends inside the kernels, without launch gaps.  None when the profiler is unavailable."""
    try:
        from torch.profiler import ProfilerActivity, profile
        step()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            step()
            torch.cuda.synchronize()
        tot = 0.0
        for e in prof.key_averages():
            if "memcpy" in e.key.lower() or "memset" in e.key.lower():
                continue
            tot += float(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)))
        return tot / 1e3 if tot > 0 else None
    except Exception:  # noqa: BLE001
        return None


def reference_gpu(torch, model, make_inputs, device, steps, lib=None):
    """The reference's own CUDA kernels (oracle/_ref: unmodified sources rebuilt for sm_100a) through their own entry
    points: plain launches on the legacy default stream (they cannot be graph-captured), and the kernel-only device
    time of the same step.  With `lib`, this repo's C ABI is timed in the SAME two modes beside it."""
    d = os.path.join(ROOT, "oracle", "_ref")
    sys.path.insert(0, d)
    import importlib
    ref = importlib.import_module("ref_awq_engine")
    out = {}
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    for tag, M, k in (("decode", 1, steps), ("prefill", 2048, 5)):
        xs = make_inputs(M, 0.25)
        ys = {N: torch.empty(M, N, dtype=torch.float16, device=device) for N in {m["N"] for m in model}}

        def step():
            for m in model:
                if M < 8:
                    ref.gemv_forward_cuda_new(xs[m["K"]], m["qw"], m["sc"], m["sz"], M, m["N"], m["K"], G)
                else:
                    ref.gemm_forward_cuda_new(xs[m["K"]], m["qw"], m["sc"], m["sz"])

        def ours():
            st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            for m in model:
                a = (p(xs[m["K"]]), p(m["qw"]), p(m["sc"]), p(m["sz"]), p(ys[m["N"]]), M, m["N"], m["K"], G, 0)
                rc = lib.b200awq_w4a16_gemv(*a, st) if M < 8 else lib.b200awq_w4a16_gemm(*a, None, 0, st)
                if rc != 0:
                    raise RuntimeError(lib.b200awq_strerror(rc).decode())
        with torch.cuda.stream(torch.cuda.default_stream()):
            ms, _ = timed_steps(torch, None, device, step, k, 3)
            ko = kernel_only_ms(torch, step)
        out[tag] = {"value": M * 1000.0 * k / ms, "unit": UNIT, "ms_per_step": ms / k, "steps": k,
                    "eager": {"value": M * 1000.0 * k / ms, "ms_per_step": ms / k},
                    "kernel_only": None if ko is None else {"value": M * 1000.0 / ko, "ms_per_step": ko}}
        if lib is not None:
            ms_o, _ = timed_steps(torch, None, device, ours, k, 3)
            # kernel-only needs non-overlapping kernels: with programmatic dependent launch a kernel's device duration
            # includes the time it spends prefetching under its predecessor, so the durations are summed with PDL off
            prev = lib.b200awq_set_pdl(0)
            ms_np, _ = timed_steps(torch, None, device, ours, k, 3)
            ko_o = kernel_only_ms(torch, ours)
            lib.b200awq_set_pdl(prev)
            out[tag]["this_repo_same_modes"] = {
                "eager": {"value": M * 1000.0 * k / ms_o, "ms_per_step": ms_o / k},
                "eager_pdl_off": {"value": M * 1000.0 * k / ms_np, "ms_per_step": ms_np / k},
                "kernel_only_pdl_off": None if ko_o is None else {"value": M * 1000.0 / ko_o, "ms_per_step": ko_o}}
    out["how"] = ("ref_awq_engine.{gemv,gemm}_forward_cuda_new, 160 calls per step: `eager` = plain launches timed with CUDA "
                  "events, `kernel_only` = sum of kernel device durations (CUPTI); this_repo_same_modes = this repo's C ABI "
                  "in the same modes (plain launches, no CUDA graph; kernel-only with programmatic dependent launch off, because overlapped "
                  "kernels' durations cannot be summed)")
    return out


def run_reference(args):
    """Reference arm: the reference has no CPU implementation of this path (CUDA only), so the CPU arm is
    the oracle port of its pure-PyTorch dequant formula on all host threads.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    step = cpu_layer(torch)
    pick_cpu_threads(torch, step)
    for _ in range(max(args.warmup, 1)):
        step()
    steps = min(args.steps, args.cpu_steps)
    t0 = time.time()
    for _ in range(steps):
        step()
    dt = (time.time() - t0) / steps
    v = 1.0 / (dt * LLAMA3_8B["layers"])
    sample = "each step = 1 of 32 decoder layers (5 WQLinear forwards, M=1, dequant every call); tok/s = 1/(32 x step time)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC % max(int(args.gpus), 1), "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": max(args.warmup, 1),
        "ms_per_step": dt * 1e3, "steps_per_token": LLAMA3_8B["layers"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32",
        "data": "synthetic", "config": {"workload": "Llama-3-8B W4A16 g128 decode bs=1 (BASELINE configs[1]), CPU pure-PyTorch dequant path",
                                        "sample": sample},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "host_cores": os.cpu_count(), "kind": "port",
                         "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


def run_reference_gpu(args):
    import torch
    if int(os.environ.get("RANK", "0")) != 0:
        return
    device = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    model = build_model(torch, LLAMA3_8B, torch.float16, device)

    def make_inputs(M, scale=1.0):
        g = torch.Generator(device=device).manual_seed(99 + M)
        return {K: (torch.randn(M, K, generator=g, device=device) * scale).to(torch.float16) for K in (4096, 14336)}
    r = reference_gpu(torch, model, make_inputs, device, args.steps)
    print(json.dumps({"impl": "reference-gpu", "metric": METRIC % 1, "value": r["decode"]["value"], "unit": UNIT, "n_gpus": 1,
                      "higher_is_better": True, "detail": r}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=500,
                    help="timed steps of each GPU leg (the reference kernels' prefill comparison times 5; "
                         "--impl reference times min(--steps, --cpu-steps) on the host)")
    ap.add_argument("--warmup", type=int, default=10, help="untimed steps before each leg of --impl b200")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "reference-gpu"])
    ap.add_argument("--prefill-steps", type=int, default=None, help="timed prefill steps instead of --steps")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--cpu-steps", type=int, default=30)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-ref-gpu", dest="ref_gpu", action="store_false")
    ap.add_argument("--no-sweep", dest="sweep", action="store_false")
    ap.add_argument("--workload", default="llama3", choices=["llama3", "tp70b"])
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step of each leg as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "b200" or args.workload != "llama3"):
        ap.error("--dump-outputs writes the outputs of --impl b200 --workload llama3 only")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-gpu":
        run_reference_gpu(args)
    elif args.workload == "tp70b":
        run_tp70b(args)
    else:
        run_b200(args)
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.destroy_process_group()
    except Exception:  # noqa: BLE001
        pass


if __name__ == "__main__":
    main()
