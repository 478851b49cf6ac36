"""torchrun worker: expert-parallel MoE (fused dispatch/combine over peer memory) == local MoE."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

from mlx_sharding_b200.ops import b200, reference as R  # noqa: E402
from mlx_sharding_b200.ops.weights import LinearWeight  # noqa: E402
from mlx_sharding_b200.parallel.ep import EPBuffers, ExpertParallelMoE  # noqa: E402

if __name__ == "__main__":
    lr = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    rank, world = dist.get_rank(), dist.get_world_size()
    H, I, E, k, T = 2048, 1408, 64, 6, 48
    g = torch.Generator(device="cuda").manual_seed(5)            # identical weights on every rank
    mk = lambda *s, sc=0.03: (torch.randn(*s, device="cuda", generator=g) * sc).to(torch.bfloat16)
    Wg, Wu, Wd, gate = LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, H, I)), mk(E, H, sc=0.05)
    g2 = torch.Generator(device="cuda").manual_seed(100 + rank)  # different tokens per rank
    x = torch.randn(T, H, device="cuda", generator=g2).to(torch.bfloat16)
    res = torch.randn(T, H, device="cuda", generator=g2).to(torch.bfloat16)
    idx, w = b200.moe_route(x, gate, k)
    bufs = EPBuffers(H, 64, k, experts_per_rank=E // world)
    ep = ExpertParallelMoE(bufs, Wg, Wu, Wd, E)
    ok = True
    for it in range(3):  # several rounds: buffer reuse + counting flags
        got = ep.forward(x, idx, w, residual=res)
        torch.cuda.synchronize()
        ref = b200.moe_experts(x, idx, w, Wg, Wu, Wd, "silu", residual=res)
        err = (got.float() - ref.float()).abs().max().item()
        ok = ok and err < 2e-2 and not bufs.error()
        dist.barrier()
    # CUDA-graph replay of the whole EP layer
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        out_g = ep.forward(x, idx, w, residual=res)
    for _ in range(3):
        gr.replay()
    torch.cuda.synchronize()
    err_g = (out_g.float() - ref.float()).abs().max().item()
    ok = ok and err_g < 2e-2 and not bufs.error()
    flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"max err {err:.4g} graph {err_g:.4g}")
        if flag.item() == 1.0:
            print("EP_OK")
    dist.barrier()
    dist.destroy_process_group()
