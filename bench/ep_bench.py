#!/usr/bin/env python
"""BASELINE config 5: DeepSeek-Coder-V2-Lite MoE blocks with the fused expert all-to-all (expert parallelism).

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 bench/ep_bench.py [--tokens 64]

Every rank routes its own ``--tokens`` tokens through one MoE block (router -> 6 of 64 experts -> weighted combine):

* ``local``: all 64 experts resident on the rank (what a pipeline stage does today) — the rank streams the whole
  1.1 GB expert bank per block;
* ``ep``   : experts sharded over the N ranks (64/N each); tokens travel through the fused dispatch / return kernels
  over NVLink peer memory (``ops/csrc/ep.cu``) — each rank streams 1/N of the bank but serves N x tokens.

Prints one JSON line (rank 0): device-timed microseconds per block (CUDA graph of ``--layers`` chained blocks, max over
ranks), aggregate tokens/s per block, NVLink bytes per block and the achieved fraction of the roofline
max(weight-stream time at measured HBM bandwidth, NVLink bytes / 770 GB/s).
"""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from mlx_sharding_b200.ops import b200  # noqa: E402
from mlx_sharding_b200.ops.weights import LinearWeight  # noqa: E402
from mlx_sharding_b200.parallel.ep import EPBuffers, ExpertParallelMoE  # noqa: E402
from mlx_sharding_b200.utils.timing import max_over_ranks  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tokens", type=int, default=64, help="tokens per rank per step")
    ap.add_argument("--layers", type=int, default=8, help="chained MoE blocks inside the timed graph")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--breakdown", action="store_true", help="also print an eager per-phase timing of one EP block (CUDA events)")
    args = ap.parse_args()
    lr = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(lr)
    dist.init_process_group("nccl", device_id=torch.device("cuda", lr))
    rank, world = dist.get_rank(), dist.get_world_size()
    H, I, E, k, T = 2048, 1408, 64, 6, args.tokens
    g = torch.Generator(device="cuda").manual_seed(5)
    mk = lambda *s, sc=0.03: (torch.randn(*s, device="cuda", generator=g) * sc).to(torch.bfloat16)
    L = args.layers
    banks = [(LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, I, H)), LinearWeight(weight=mk(E, H, I)), mk(E, H, sc=0.05))
             for _ in range(L)]
    g2 = torch.Generator(device="cuda").manual_seed(100 + rank)
    x0 = torch.randn(T, H, device="cuda", generator=g2).to(torch.bfloat16)
    bufs = EPBuffers(H, max(T, 64), k, experts_per_rank=E // world)
    eps = [ExpertParallelMoE(bufs, Wg, Wu, Wd, E) for (Wg, Wu, Wd, _) in banks]

    def run_local(x):
        for (Wg, Wu, Wd, gate) in banks:
            idx, w = b200.moe_route(x, gate, k)
            x = b200.moe_experts(x, idx, w, Wg, Wu, Wd, "silu", residual=x)
        return x

    def run_ep(x):
        for ep, (_, _, _, gate) in zip(eps, banks):
            idx, w = b200.moe_route(x, gate, k)
            x = ep.forward(x, idx, w, residual=x)
        return x

    def timed(fn):
        for _ in range(2):
            fn(x0)
        torch.cuda.synchronize()
        dist.barrier()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            out = fn(x0)
        gr.replay()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            gr.replay()
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        return max_over_ranks(e0.elapsed_time(e1)) * 1e3 / (args.iters * L), out

    if args.breakdown:
        # eager, event-timed phases of one EP block on this rank, the calls of ExpertParallelMoE.forward (launch gaps included; the
        # arrival wait shows up in gate_up, the return wait in combine)
        ep, (_, _, _, gate) = eps[0], banks[0]
        b, C, W = bufs, bufs.C, world
        names = ["route", "dispatch", "gate_up(+arrival wait)", "down(+return)", "combine(+wait)"]
        acc = [0.0] * len(names)
        n_it = 20
        exp_rows = T * k
        stride = b.stride(T)
        rows, row_dst = b.recv_views(stride)
        mr = min(W * T, stride)
        arrive = (stride, b.base + b.off_recv_count, b.seq, b.error_ptr, W)
        for it in range(n_it + 3):
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(len(names) + 1)]
            dist.barrier()
            evs[0].record()
            idx, w = b200.moe_route(x0, gate, k); evs[1].record()
            C.ep_dispatch_scatter(x0, idx, ep.E_local, b.rank, stride, b.t_recv_x, b.t_recv_meta, b.t_cnt, b.t_recv_count, b.t_my_ret,
                                  b.seq, b.done, b.ret_expected); evs[2].record()
            h = C.grouped_linear(rows, ep.wg, ep.wu, b.cnt, mr, ep.act, False, None, None, None, exp_rows, *arrive, True); evs[3].record()
            C.grouped_linear(h, ep.wd, None, b.cnt, mr, 0, True, row_dst, b.ret_flags_dev, b.tiles, exp_rows, *arrive, False)
            evs[4].record()
            C.ep_combine(b.base + b.off_flags + 128, b.ret_expected, b.error_ptr, b.ret_y, w, x0, None); evs[5].record()
            torch.cuda.synchronize()
            if it >= 3:
                for i in range(len(names)):
                    acc[i] += evs[i].elapsed_time(evs[i + 1]) * 1e3 / n_it
        print(f"[rank {rank}] eager EP block phases (us): " + ", ".join(f"{n} {v:.1f}" for n, v in zip(names, acc)) + f"  total {sum(acc):.1f}",
              file=sys.stderr, flush=True)
        dist.barrier()

    us_local, out_l = timed(run_local)
    us_ep, out_e = timed(run_ep)
    # correctness on ONE block (the chained blocks of the timed graphs are not normalised, their values overflow)
    (Wg, Wu, Wd, gate) = banks[0]
    idx, w = b200.moe_route(x0, gate, k)
    ref1 = b200.moe_experts(x0, idx, w, Wg, Wu, Wd, "silu", residual=x0)
    got1 = eps[0].forward(x0, idx, w, residual=x0)
    torch.cuda.synchronize()
    err = (ref1.float() - got1.float()).abs().max().item()
    bank_bytes = 3 * E * I * H * 2
    nvl_bytes = T * k * (world - 1) / world * (H * 2 + H * 4)          # dispatch bf16 + return fp32, remote share
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm = peaks.get("hbm_gbs", 6650.0) * 1e9
    roof_us = max(bank_bytes / world / hbm, nvl_bytes / 770e9) * 1e6
    if rank == 0:
        print(json.dumps({
            "bench": "DeepSeek-V2-Lite MoE block, expert parallel fused all-to-all", "n_gpus": world, "tokens_per_rank": T,
            "us_per_block_local": round(us_local, 2), "us_per_block_ep": round(us_ep, 2),
            "tokens_per_s_local": round(world * T / us_local * 1e6), "tokens_per_s_ep": round(world * T / us_ep * 1e6),
            "speedup_ep_vs_local": round(us_local / us_ep, 3), "nvlink_bytes_per_block_per_rank": int(nvl_bytes),
            "roofline_us": round(roof_us, 2), "roofline_fraction": round(roof_us / us_ep, 3),
            "roofline_basis": f"max(expert bank / N at {'measured' if peaks else 'fallback'} HBM {hbm / 1e9:.0f} GB/s, NVLink bytes at 770 GB/s)",
            "max_abs_diff_vs_local": err, "p2p_error": bool(bufs.error())}), flush=True)
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
