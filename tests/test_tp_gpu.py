"""Tensor-parallel modules on real kernels + NCCL (needs >= 2 GPUs)."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu


def _worker(rank, world, port, out_dir):
    import llm_awq_b200 as P
    from llm_awq_b200 import tp
    from awq_testutil import gen_layer, gen_x
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    dev = f"cuda:{rank}"
    hidden, inter = 1024, 2048

    def full(N, K, seed, bias):
        m = P.WQLinear(4, 128, K, N, bias, "cpu")
        m.qweight, m.scales, m.scaled_zeros = gen_layer(N, K, torch.float16, seed=seed)
        if bias:
            m.bias = torch.randn(N, generator=torch.Generator().manual_seed(seed + 100)).half()
        return m
    up, down = full(inter, hidden, 1, False), full(hidden, inter, 2, True)
    col = tp.ColumnParallelWQLinear(up, rank, world).to(dev)
    row = tp.RowParallelWQLinear(down, rank, world).to(dev)
    row.bias = row.bias.to(dev)
    ex = tp.PeerExchange(8, hidden)
    fused = tp.FusedRowParallelWQLinear(down, rank, world, ex).to(dev)
    fused.bias = fused.bias.to(dev)
    outs = {}
    for M in (1, 5, 33):
        x = gen_x(M, hidden, seed=M).to(dev)
        h = col(x)                 # [M, inter / world] on this rank
        y = row(h)                 # local kernel + ONE all-reduce + bias
        yf = [fused(h).cpu() for _ in range(3)]      # fused GEMV + NVLink exchange (M <= 8), repeated (epochs)
        outs[M] = (h.cpu(), y.cpu(), yf)
    # CUDA-graph replay of the fused kernel (epochs live on the device)
    hs = col(gen_x(2, hidden, seed=2).to(dev)).clone()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        fused(hs)
    s.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        yg = fused(hs)
    reps = []
    for _ in range(4):
        g.replay()
        torch.cuda.synchronize()
        reps.append(yg.cpu().clone())
    outs["graph"] = (reps, row(hs).cpu())
    torch.save(outs, os.path.join(out_dir, f"r{rank}.pt"))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.multigpu
def test_column_then_row_parallel_on_kernels_nccl(tmp_path):
    from oracle import w4a16_oracle as O
    from awq_testutil import gen_layer, gen_x, np64, rel_err
    world = 2
    mp.spawn(_worker, args=(world, 29600 + os.getpid() % 300, str(tmp_path)), nprocs=world, join=True)
    outs = [torch.load(os.path.join(tmp_path, f"r{r}.pt")) for r in range(world)]
    hidden, inter = 1024, 2048
    uq, us, uz = gen_layer(inter, hidden, torch.float16, seed=1)
    dq, ds, dz = gen_layer(hidden, inter, torch.float16, seed=2)
    bias = torch.randn(hidden, generator=torch.Generator().manual_seed(102)).half()
    for M in (1, 5, 33):
        x = gen_x(M, hidden, seed=M)
        h64 = O.wq_linear_forward(np64(x), uq.numpy(), np64(us), np64(uz))
        h = torch.cat([outs[r][M][0] for r in range(world)], dim=1)            # column shards concatenate
        assert rel_err(np64(h), h64) < 1e-3
        y64 = O.wq_linear_forward(np64(h), dq.numpy(), np64(ds), np64(dz), bias=np64(bias))
        for r in range(world):
            assert torch.equal(outs[r][M][1], outs[0][M][1])                   # all ranks hold the reduced result
        assert rel_err(np64(outs[0][M][1]), y64) < 2e-3                        # two fp16 roundings (partials, bias add)
        for yf in outs[0][M][2]:                                                # fused path: fp32 partials, one rounding
            assert rel_err(np64(yf), y64) < 1e-3
        for r in range(world):
            for a, b in zip(outs[r][M][2], outs[0][M][2]):
                assert torch.equal(a, b)                                        # bit-identical across ranks and repeats
    reps, ref = outs[0]["graph"]
    for rr in reps:
        assert torch.equal(rr, reps[0]) and rel_err(np64(rr), np64(ref)) < 1e-3
