"""torchrun worker: expert-parallel MoE under the conditions of a whole model — several layers sharing one ``EPBuffers`` called
back to back with no host synchronisation in between, token counts that change from step to step (prefill chunk -> decode
batch -> ...), two geometries (DeepSeek-V2-Lite's and the tiny test model's) — every output compared against the local MoE.
``argv[1]``: ``forward`` (rows routed separately, then ``ExpertParallelMoE.forward``) or ``fused`` (``route_forward``).  Prints
one line per (geometry, step) and ``EP_STRESS_OK <mode>`` on rank 0."""
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

from mlx_sharding_b200.ops import b200  # noqa: E402
from mlx_sharding_b200.ops.weights import LinearWeight  # noqa: E402
from mlx_sharding_b200.parallel.ep import EPBuffers, ExpertParallelMoE  # noqa: E402


def run_fused(H, I, E, k, Ts, layers, rank, world):
    """``route_forward``: [norm + router + dispatch] -> GEMMs -> [combine + next norm], against separate norm / route / local experts."""
    g = torch.Generator(device="cuda").manual_seed(5)
    mk = lambda *s, sc=0.03: (torch.randn(*s, device="cuda", generator=g) * sc).to(torch.bfloat16)
    banks = [(LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, H, I)), mk(E, H, sc=0.05),
              (1.0 + mk(H, sc=3.0)).contiguous(), (1.0 + mk(H, sc=3.0)).contiguous()) for _ in range(layers)]
    maxT = max(Ts)
    bufs = EPBuffers(H, maxT, k, experts_per_rank=E // world)
    eps = [ExpertParallelMoE(bufs, b[0], b[1], b[2], E) for b in banks]
    rk = dict(top_k=k, method="greedy", n_group=1, topk_group=1, scaling=1.0, norm_topk=False)
    g2 = torch.Generator(device="cuda").manual_seed(200 + rank)
    ok = True
    for step, T in enumerate(Ts):
        hs = [(torch.randn(T, H, device="cuda", generator=g2) * 2.0).to(torch.bfloat16) for _ in range(layers)]
        torch.cuda.synchronize()
        outs = [ep.route_forward(h, b[3], rk, (b[4], 1e-6), (lambda h_: (lambda normed: (h_, None)))(h), next_norm=(b[5], 1e-6))
                for ep, h, b in zip(eps, hs, banks)]                                                         # back to back
        torch.cuda.synchronize()
        worst, badrows, rows = 0.0, 0, 0
        for (Wg, Wu, Wd, gate, n1, n2), h, (got, got_n) in zip(banks, hs, outs):
            normed = b200.rmsnorm(h, n1, 1e-6)
            idx, w = b200.moe_route(normed, gate, k)
            ref = b200.moe_experts(normed, idx, w, Wg, Wu, Wd, "silu", residual=h)
            ref_n = b200.rmsnorm(ref, n2, 1e-6)
            # per-row error relative to the row's magnitude (the test's norm weights make the values large: one bf16 ulp of an
            # output near 32 is 0.25)
            rel = lambda a, b_: (a.float() - b_.float()).abs().amax(-1) / (b_.float().abs().amax(-1) + 1.0)
            d = torch.maximum(rel(got, ref), rel(got_n, ref_n))
            worst = max(worst, d.max().item())
            badrows += int((d > 2e-2).sum().item())
            rows += T
        # a normalised value may land on the neighbouring bf16 (statistics summed in a different order), which can flip a near-tie
        # of the router for a rare token: tolerate one such row per step, nothing systematic
        good = badrows <= 1 and not bufs.error()
        ok = ok and good
        print(f"[rank {rank}] fused H={H} E={E} step {step} T={T}: max rel err {worst:.4g}, bad rows {badrows}/{rows}, error flag {bufs.error()}", flush=True)
    return ok


def run(H, I, E, k, Ts, layers, rank, world):
    g = torch.Generator(device="cuda").manual_seed(5)
    mk = lambda *s, sc=0.03: (torch.randn(*s, device="cuda", generator=g) * sc).to(torch.bfloat16)
    banks = [(LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, H, I)), mk(E, H, sc=0.05))
             for _ in range(layers)]
    maxT = max(Ts)
    bufs = EPBuffers(H, maxT, k, experts_per_rank=E // world)
    eps = [ExpertParallelMoE(bufs, Wg, Wu, Wd, E) for Wg, Wu, Wd, _ in banks]
    g2 = torch.Generator(device="cuda").manual_seed(100 + rank)
    ok = True
    for step, T in enumerate(Ts):
        xs = [torch.randn(T, H, device="cuda", generator=g2).to(torch.bfloat16) for _ in range(layers)]
        rs = [torch.randn(T, H, device="cuda", generator=g2).to(torch.bfloat16) for _ in range(layers)]
        routes = [b200.moe_route(x, bank[3], k) for x, bank in zip(xs, banks)]
        torch.cuda.synchronize()
        outs = [ep.forward(x, idx, w, residual=r) for ep, x, (idx, w), r in zip(eps, xs, routes, rs)]   # back to back
        torch.cuda.synchronize()
        worst, badrows = 0.0, 0
        for (Wg, Wu, Wd, _), x, (idx, w), r, got in zip(banks, xs, routes, rs, outs):
            ref = b200.moe_experts(x, idx, w, Wg, Wu, Wd, "silu", residual=r)
            d = (got.float() - ref.float()).abs().amax(-1)
            worst = max(worst, d.max().item())
            badrows += int((d > 2e-2).sum().item())
        good = worst < 2e-2 and not bufs.error()
        ok = ok and good
        print(f"[rank {rank}] H={H} E={E} step {step} T={T}: max err {worst:.4g}, bad rows {badrows}, error flag {bufs.error()}", flush=True)
    # the same layers inside one CUDA graph, replayed
    T = Ts[-1]
    xs = [torch.randn(T, H, device="cuda", generator=g2).to(torch.bfloat16) for _ in range(layers)]
    routes = [b200.moe_route(x, bank[3], k) for x, bank in zip(xs, banks)]
    for ep, x, (idx, w) in zip(eps, xs, routes):
        ep.forward(x, idx, w)
    torch.cuda.synchronize()
    dist.barrier()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        outs = [ep.forward(x, idx, w) for ep, x, (idx, w) in zip(eps, xs, routes)]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(5):
        gr.replay()
    torch.cuda.synchronize()
    dist.barrier()
    ev[0].record()
    for _ in range(20):
        gr.replay()
    ev[1].record()
    torch.cuda.synchronize()
    us = ev[0].elapsed_time(ev[1]) * 1e3 / 20 / layers
    worst = 0.0
    for (Wg, Wu, Wd, _), x, (idx, w), got in zip(banks, xs, routes, outs):
        ref = b200.moe_experts(x, idx, w, Wg, Wu, Wd, "silu")
        worst = max(worst, (got.float() - ref.float()).abs().max().item())
    ok = ok and worst < 2e-2 and not bufs.error()
    print(f"[rank {rank}] H={H} E={E} graph T={T}: max err {worst:.4g}, {us:.1f} us per EP layer", flush=True)
    return ok


if __name__ == "__main__":
    lr = int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(lr)
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    rank, world = dist.get_rank(), dist.get_world_size()
    mode = sys.argv[1] if len(sys.argv) > 1 else "forward"
    check = run_fused if mode == "fused" else run
    ok = check(256, 128, 8, 3, [384, 16, 16, 48, 384, 16], 3, rank, world)
    ok = check(2048, 1408, 64, 6, [256, 64, 64, 48, 256, 64], 5, rank, world) and ok
    flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0 and flag.item() == 1.0:
        print("EP_STRESS_OK", mode)
    dist.barrier()
    dist.destroy_process_group()
