#!/usr/bin/env python
"""Headline benchmark (BASELINE.json): decode tokens/sec (+ p50 TTFT) of DeepSeek-Coder-V2-Lite on N B200s.

    python bench.py --gpus 1 --steps 32 --warmup 4
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

* model   : DeepSeek-Coder-V2-Lite-Instruct architecture (27 layers, 64 routed experts top-6, MLA), bf16,
            random-init weights in the mlx-community layout, synthetic prompts (the box is offline).
* sharding: on N > 1 GPUs two shardings of the model are measured in the same run (``--parallelism auto``) and the faster
            one is the headline, the other is reported under ``also_measured``:
            pp — N pipeline stages (cost-balanced layer / half-layer ranges), N micro-batch groups of ``--batch`` sequences in
                 flight, fused P2P stage hand-off (the reference's layer-range sharding, BASELINE config 3);
            ep — every rank decodes its own ``--batch`` sequences through all layers (attention replicated) and holds E/N routed
                 experts of every MoE layer, exchanged with the fused all-to-all over NVLink peer memory (BASELINE config 5).
            Both are weak scaling: per-GPU work is fixed, global batch = N x batch.
* step    : one decode step of every sequence in flight = ``N * batch`` new tokens.  ``value`` = whole-job tokens/sec,
            device-timed with CUDA events after ``--warmup`` steps, max over ranks.
* e2e     : the same metric through the public serving API (``LLMEngine.submit/step``): every step copies
            the step's token ids + metadata host->device from pinned memory and reads the sampled tokens
            back device->host.
* --impl reference : the unmodified mzbac/mlx_sharding from ``baseline/_ref`` (needs Apple's ``mlx``; reports
            ``unavailable`` on this platform).  --impl baseline : the same pipeline as plain PyTorch ops
            (cuBLAS GEMMs, eager, NCCL p2p hand-off) — the "straight re-implementation" BASELINE.md names.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse_args(argv=None):
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=32)
    p.add_argument("--warmup", type=int, default=4)
    p.add_argument("--impl", type=str, default="ours", choices=["ours", "reference", "baseline"])
    p.add_argument("--batch", type=int, default=64, help="sequences per micro-batch group (one group per stage)")
    p.add_argument("--prompt-len", type=int, default=128)
    p.add_argument("--model", type=str, default="deepseek-v2-lite", choices=["deepseek-v2-lite", "llama3-8b", "tiny"])
    p.add_argument("--transport", type=str, default="auto", choices=["auto", "fused", "nccl"])
    p.add_argument("--layers", type=int, default=None, help="debug only: truncate the model (result is marked invalid)")
    p.add_argument("--groups", type=int, default=0, help="micro-batch groups in flight (default: one per stage)")
    p.add_argument("--quant", type=int, default=0, choices=[0, 4, 8],
                   help="MLX affine quantised weights (group 64), dequantised inside the GEMM kernels (BASELINE config 2)")
    p.add_argument("--fp8-experts", action="store_true",
                   help="convert the routed / shared expert banks to block-scaled MXFP8 at load (tcgen05 kind::mxf8f6f4); this is the "
                        "default for --quant 4/8 checkpoints (MLXB200_FP8_EXPERTS=0 keeps the exact in-kernel MLX-affine dequant)")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-baseline", action="store_true",
                   help="skip the short same-box baseline run (baseline/torch_pipeline.py) that fills vs_baseline")
    p.add_argument("--baseline-steps", type=int, default=8)
    p.add_argument("--no-graphs", action="store_true")
    p.add_argument("--page-size", type=int, default=64)
    p.add_argument("--whole-layers", action="store_true", help="stage boundaries only between layers (reference-style split)")
    p.add_argument("--parallelism", type=str, default="auto", choices=["auto", "pp", "ep"],
                   help="auto (default): pp on 1 GPU / dense models; on N>1 GPUs with an MoE model measure pp AND ep and headline the "
                        "faster, reporting the other under 'also_measured'.  "
                        "pp: layer-range pipeline, one micro-batch group per stage (the reference's sharding).  "
                        "ep: every rank runs all layers on its own --batch sequences (data-parallel attention) and the routed "
                        "experts of every MoE layer are sharded over the ranks with the fused all-to-all (BASELINE config 5)")
    p.add_argument("--dump-outputs", type=str, default=None, metavar="DIR",
                   help="after the timed decode steps, write what the last step returned as DIR/<name>.npy: the sampled token ids "
                        "(float64) and the fp32 logits of every sequence, at most 64 MB in all (logits that do not fit keep a fixed, "
                        "seeded subset of vocabulary columns).  Inputs are seeded, so two builds run with the same arguments can be "
                        "compared output for output")
    args = p.parse_args(argv)
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs records the outputs of --impl ours")
    return args


def reference_arm(args):
    """Run the UNMODIFIED reference from baseline/_ref through its own API — or say why that is impossible."""
    ref = os.path.join(ROOT, "baseline", "_ref")
    out = {"impl": "reference"}
    if not os.path.isdir(os.path.join(ref, "shard")):
        out["unavailable"] = "baseline/_ref is not installed (pip install --no-deps --target baseline/_ref /root/reference)"
    else:
        sys.path.insert(0, ref)
        try:
            import importlib

            importlib.import_module("shard.utils")  # imports mlx.core / mlx_lm at module scope
            out["unavailable"] = "reference imported but has no CUDA execution path (MLX Metal only)"
        except Exception as e:  # noqa: BLE001
            out["unavailable"] = (f"reference needs Apple MLX: {type(e).__name__}: {e} "
                                  "(mlx / mlx_lm have no Linux+CUDA wheel in the offline wheelhouse)")
        finally:
            sys.path.remove(ref)
    if int(os.environ.get("RANK", "0")) == 0:
        print(json.dumps(out), flush=True)
    return 0


def model_config(name: str, layers=None):
    from mlx_sharding_b200.config import deepseek_v2_lite_config, llama3_8b_config

    if name == "deepseek-v2-lite":
        cfg = deepseek_v2_lite_config()
    elif name == "llama3-8b":
        cfg = llama3_8b_config()
    else:
        cfg = dict(deepseek_v2_lite_config(), hidden_size=256, num_hidden_layers=4, num_attention_heads=2,
                   num_key_value_heads=2, kv_lora_rank=64, moe_intermediate_size=128, n_routed_experts=8,
                   num_experts_per_tok=3, intermediate_size=512, vocab_size=512)
    if layers:
        cfg["num_hidden_layers"] = layers
    return cfg


def main(argv=None):
    args = parse_args(argv)
    if args.impl == "reference":
        return reference_arm(args)
    if args.fp8_experts:
        os.environ["MLXB200_FP8_EXPERTS"] = "1"

    import gc

    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", str(rank)))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)

    if args.impl == "baseline":
        # same-box baseline arm: plain PyTorch (cuBLAS + SDPA, CUDA-graphed stage steps) + NCCL p2p — baseline/torch_pipeline.py
        from baseline.torch_pipeline import run as run_baseline

        res = run_baseline(args, world, rank, local, dev, e2e=not args.no_e2e)
        if rank == 0:
            print(json.dumps(res), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return 0

    # a short run of the baseline arm in the same process, on the same GPUs, right before the product: fills ``vs_baseline``
    base = None
    if not args.no_baseline:
        try:
            from baseline.torch_pipeline import run as run_baseline

            base = run_baseline(args, world, rank, local, dev, steps=max(1, min(args.steps, args.baseline_steps)), warmup=3,
                                e2e=not args.no_e2e)
        except Exception:  # noqa: BLE001 — the product measurement does not depend on the baseline arm
            import traceback

            traceback.print_exc()
            base = None
        gc.collect()
        torch.cuda.empty_cache()
        settle = float(os.environ.get("MLXB200_BENCH_SETTLE_S", "0") or 0)
        if settle > 0:
            time.sleep(settle)
        if world > 1:
            dist.barrier()

    moe = args.model != "llama3-8b"
    mode = args.parallelism
    if mode == "auto":
        # MoE model on several GPUs: measure BOTH shardings — the layer-range pipeline (the reference's sharding, BASELINE
        # config 3) and expert parallelism with the fused all-to-all (config 5) — and headline the faster one
        mode = "both" if (world > 1 and moe and args.impl == "ours" and not args.quant) else "pp"
    if mode == "ep" and (world == 1 or not moe or args.impl != "ours"):
        mode = "pp"
    res = None
    if mode in ("pp", "both"):
        res = run_pp(args, world, rank, local, dev)
    if mode in ("ep", "both"):
        gc.collect()
        torch.cuda.empty_cache()
        try:
            ep = run_ep(args, world, rank, local, dev)
        except Exception:  # noqa: BLE001 — keep the pipeline measurement if the second sharding fails on every rank
            import traceback

            traceback.print_exc()
            if mode != "both":   # nothing else was measured
                raise
            ep = None
            if rank == 0 and res is not None:
                res["also_measured"] = {"expert parallel (config 5)": {"error": "run failed, see stderr"}}
        if rank == 0 and ep is not None:
            res = merge_results(res, ep)
    if rank == 0:
        print(json.dumps(attach_baseline(res, base)), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def weights_desc(args) -> str:
    fp8 = os.environ.get("MLXB200_FP8_EXPERTS", "")
    if args.quant:
        exp = "expert banks converted to block-scaled MXFP8 at load (tcgen05 kind::mxf8f6f4)" if fp8 != "0" else "expert banks dequantised in-kernel"
        return f"mlx-affine-int{args.quant}-g64 checkpoint: attention / dense weights dequantised in-kernel, {exp}"
    return "bf16" + (", expert banks converted to block-scaled MXFP8 at load" if fp8 == "1" else "")


METRIC = "decode tokens/sec, DeepSeek-Coder-V2-Lite @N B200, + p50 TTFT"


def attach_baseline(res, base):
    """``vs_baseline`` = value / the same-box baseline arm measured in this run (BASELINE.md publishes no number; the baseline to
    beat is "a straight PyTorch cuBLAS + SDPA + NCCL-p2p re-implementation measured on the same box").  Pure function, unit-tested."""
    if res is None:
        return res
    if not base or not base.get("value"):
        res["vs_baseline"] = None
        return res
    ratio = lambda a, b: round(a / b, 3) if (a and b) else None
    res["vs_baseline"] = ratio(res["value"], base["value"])
    b = {"impl": "baseline (baseline/torch_pipeline.py: cuBLAS + SDPA, CUDA-graphed stage steps, NCCL send/recv)",
         "value": base["value"], "ms_per_step": base["ms_per_step"], "steps": base["steps"],
         "ttft_p50_ms": base.get("ttft_p50_ms"), "ttft_microbatch_ms": base.get("ttft_microbatch_ms"),
         "parallelism": base["config"]["parallelism"]}
    be = base.get("e2e") or {}
    if be.get("value"):
        b["e2e_value"] = be["value"]
    res["baseline"] = b
    e = res.get("e2e")
    if isinstance(e, dict) and e.get("value") and be.get("value"):
        e["vs_baseline"] = ratio(e["value"], be["value"])
    if res.get("ttft_p50_ms") and base.get("ttft_p50_ms"):
        res["ttft_vs_baseline"] = ratio(base["ttft_p50_ms"], res["ttft_p50_ms"])   # > 1: the product answers sooner
    for name, other in (res.get("also_measured") or {}).items():
        if isinstance(other, dict) and other.get("value"):
            other["vs_baseline"] = ratio(other["value"], base["value"])
    return res


def merge_results(pp, ep):
    """Headline = the faster *valid* sharding; the other one is reported under ``also_measured`` (pure function, unit-tested)."""
    if pp is None:
        return ep
    keep = ("value", "ms_per_step", "config", "ttft_p50_ms", "ttft_stage_chain_ms", "ttft_microbatch_ms", "e2e", "gpu_launches", "clocks", "invalid")
    brief = lambda r: {k: r[k] for k in keep if k in r}
    if "invalid" not in ep and (ep["value"] >= pp["value"] or "invalid" in pp):
        return dict(ep, also_measured={"layer-range pipeline (config 3)": brief(pp)})
    return dict(pp, also_measured={"expert parallel (config 5)": brief(ep)})


DUMP_BYTES = 64_000_000


def decode_outputs(loop, prefix=""):
    """What the last decode step of ``loop`` handed back on this rank, one row per sequence of every group: the sampled token
    ids (held by the first stage, where they feed the next step) and the logits (computed by the last stage)."""
    import torch

    out = {}
    if loop.first:
        toks = [loop.p2p.token_inbox(g, loop.B) if loop.transport == "fused" else loop.groups[g].tokens for g in range(loop.G)]
        out[prefix + "tokens"] = torch.stack(toks)
    if loop.last:
        out[prefix + "logits"] = torch.stack(loop._outs)
    return out


def dump_outputs(out_dir, arrays, world):
    """Write ``name -> tensor`` as ``out_dir/<name>.npy``: token ids as float64 (exact), the rest as float32.  A run writes at
    most ``world + 1`` logits arrays (pp: the last stage's; ep: one per rank), so each gets that share of ``DUMP_BYTES``
    (less 1 MB for the token ids); a larger one keeps a fixed, seeded subset of its last-axis columns."""
    import numpy as np

    budget = (DUMP_BYTES - 1_000_000) // (world + 1)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = t.detach().cpu().numpy().astype(np.float32 if t.is_floating_point() else np.float64)
        if a.nbytes > budget:
            keep = budget // (a.nbytes // a.shape[-1])
            a = a[..., np.sort(np.random.default_rng(0).choice(a.shape[-1], keep, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_pp(args, world, rank, local, dev):
    """Layer-range pipeline: one stage per GPU, one micro-batch group per stage in flight, fused P2P hand-off."""
    import torch
    import torch.distributed as dist

    from mlx_sharding_b200.config import ModelConfig
    from mlx_sharding_b200.engine.core import LLMEngine
    from mlx_sharding_b200.engine.sampler import SamplingParams
    from mlx_sharding_b200.ops.meta import BatchMeta
    from mlx_sharding_b200.parallel.decode_loop import DecodeLoop
    from mlx_sharding_b200.parallel.partition import balanced_split
    from mlx_sharding_b200.parallel.pipeline import ChainPipeline, LocalPipeline, StageExecutor, worker_loop
    from mlx_sharding_b200.utils.loader import random_model
    from mlx_sharding_b200.utils.timing import ClockSampler, max_over_ranks

    baseline = args.impl == "baseline"
    backend = "reference" if baseline else "b200"
    if baseline:
        from mlx_sharding_b200.ops import reference as R

        R.FAST_BASELINE = True
    else:
        from mlx_sharding_b200.ops import b200

        b200.load_extension()  # fail loudly if the sm_100a extension is missing

    cfgd = model_config(args.model, args.layers)
    cfg = ModelConfig.from_dict(cfgd)
    qcfg = dict(group_size=64, bits=args.quant) if args.quant else None
    cfg.quantization = qcfg  # the partitioner's byte model follows the weight format
    # stage boundaries may fall between the attention and the MLP block of a layer (finer balance than whole layers)
    spec = balanced_split(cfg, world, half_layers=not args.whole_layers)[rank]
    t0 = time.time()
    model = random_model(cfgd, dtype=torch.bfloat16, device=dev, backend=backend, seed=1, quantization=qcfg, spec=spec)
    torch.cuda.synchronize()
    log = lambda *a: print(f"[rank {rank}]", *a, file=sys.stderr, flush=True)
    log(f"layers {spec.describe()} weights {model.weight_bytes() / 1e9:.2f} GB built in {time.time() - t0:.1f}s")

    G, B, S, PS = (args.groups or world), args.batch, args.prompt_len, args.page_size
    total_steps = args.warmup + args.steps
    e2e_steps = 0 if args.no_e2e else (args.warmup + args.steps + 2)
    max_len = S + total_steps + e2e_steps + 8
    pages_per_seq = (max_len + PS - 1) // PS
    num_pages = G * B * pages_per_seq * (1 if args.no_e2e else 2) + 1
    stage = StageExecutor(model, num_pages, PS, seed=0)

    # ------------------------------------------------------------------ prefill (eager) -> TTFT
    gen = torch.Generator().manual_seed(1234)
    prompts = torch.randint(3, cfg.vocab_size - 1, (G, B, S), generator=gen)
    bts = [[[1 + (g * B + b) * pages_per_seq + i for i in range(pages_per_seq)] for b in range(B)] for g in range(G)]
    first_tokens, ttfts = [], []
    H = cfg.hidden_size
    # TTFT = wall time from "prompt ids on the host" to "first sampled tokens of the micro-batch available",
    # through all stages.  Every group is prefilled 1 (cold, discarded) + 3 (timed) times — re-running a
    # prefill rewrites identical KV — and the p50 over all timed samples is reported.
    def chain_prefill(meta, prompt_pinned, nseq):
        """One prompt batch through every stage; returns (first tokens, wall seconds)."""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        tt = time.perf_counter()
        if rank == 0:
            x = prompt_pinned.to(dev, non_blocking=True)
        else:
            x = torch.empty(meta.num_tokens, H, dtype=torch.bfloat16, device=dev)
            dist.recv(x, rank - 1)
        out = stage.forward(x, meta)
        if rank < world - 1:
            dist.send(out, rank + 1)
            toks = torch.empty(nseq, dtype=torch.int64, device=dev)
        else:
            toks = out.argmax(-1)
        if world > 1:
            dist.broadcast(toks, world - 1)
        torch.cuda.synchronize()
        return toks, time.perf_counter() - tt

    batch_ttfts = []
    for g in range(G):
        meta = BatchMeta.build([S] * B, [0] * B, bts[g], PS, device=dev)
        prompt_pinned = prompts[g].reshape(-1).pin_memory()
        for rep in range(3):
            toks, dt = chain_prefill(meta, prompt_pinned, B)
            if rep > 0:
                batch_ttfts.append(dt)
        first_tokens.append(toks)
    # request-level TTFT: one S-token prompt arriving alone (re-prefills sequence 0 of group 0: same KV content)
    meta1 = BatchMeta.build([S], [0], [bts[0][0]], PS, device=dev)
    p1 = prompts[0, 0].pin_memory()
    for rep in range(8):
        _, dt = chain_prefill(meta1, p1, 1)
        if rep > 1:
            ttfts.append(dt)
    ttft_p50 = max_over_ranks(statistics.median(ttfts))
    ttft_batch = max_over_ranks(statistics.median(batch_ttfts))
    log(f"prefill done: TTFT p50 {ttft_p50 * 1e3:.2f} ms (1x{S} prompt), {ttft_batch * 1e3:.1f} ms for a {B}x{S} micro-batch")

    # ------------------------------------------------------------------ device-timed steady-state decode
    transport = args.transport if not baseline else "nccl"
    loop = DecodeLoop(stage, G, B, pages_per_seq, transport=transport, use_graphs=not (baseline or args.no_graphs))
    for g in range(G):
        loop.groups[g].load(torch.full((B,), S, dtype=torch.int32), torch.tensor(bts[g], dtype=torch.int32), first_tokens[g],
                            max_ctx=max_len)
    loop.warm_kernels()
    if os.environ.get("BENCH_DEBUG"):
        # stage-local time of one group step (eager, no hand-off): tells stage balance apart from scheduling
        st0 = loop.groups[0]
        xin = st0.tokens if rank == 0 else torch.zeros(B, H, dtype=torch.bfloat16, device=dev)
        for _ in range(2):
            model.forward(xin, st0.meta, stage.kv)
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(5):
            model.forward(xin, st0.meta, stage.kv)
        ev1.record()
        torch.cuda.synchronize()
        log(f"solo stage step (eager, {spec.num_local_layers} layers): {ev0.elapsed_time(ev1) / 5:.3f} ms")
    loop.capture()
    loop.prime_tokens()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    C = None if baseline else b200.C()
    for _ in range(args.warmup):
        loop.step_all()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    n_launch0 = C.launch_count() if C else 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            loop.step_all()
        e1.record()
        torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    loop.drain()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, decode_outputs(loop), world)
    p2p_err = bool(loop.p2p.error()) if loop.p2p is not None else False
    launches = (loop.launches_per_step * G * args.steps) if loop.use_graphs else ((C.launch_count() - n_launch0) if C else 0)
    ms_per_step = ms / args.steps
    tok_s = G * B * 1000.0 / ms_per_step
    log(f"decode: {ms_per_step:.3f} ms/step -> {tok_s:.0f} tok/s  (launches/step {launches / max(args.steps, 1):.0f}, p2p_err={p2p_err})")

    # ------------------------------------------------------------------ end-to-end through the public API
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, stage, world, rank, dev, cfg, prompts, G, B, S, num_pages, PS)

    if world > 1:
        dist.barrier()
    if rank == 0:
        res = {
            "metric": METRIC,
            "value": round(tok_s, 1), "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic prompts, random-init weights (mlx-community layout)",
            "impl": args.impl,
            "config": {"model": "DeepSeek-Coder-V2-Lite-Instruct" if args.model == "deepseek-v2-lite" else args.model,
                       "global_batch": G * B, "seq_len": S, "parallelism": f"pp{world}",
                       "micro_batches_in_flight": G, "tokens_per_step": G * B, "transport": loop.transport,
                       "cuda_graphs": loop.use_graphs, "kv_page_size": PS,
                       "weights": weights_desc(args),
                       "l2": "weights streamed per step (31 GB/stage-set) far exceed the 126 MB L2; no explicit flush",
                       "layers": [spec.start_layer, spec.end_layer] if world == 1 else
                       ("cost-balanced, whole layers" if args.whole_layers else "cost-balanced, half-layer (attention | MLP) boundaries")},
            "ttft_p50_ms": (e2e or {}).get("ttft_p50_ms") or round(ttft_p50 * 1e3, 3),
            "ttft_note": f"p50 over {TTFT_REQUESTS} requests through LLMEngine.submit (one {S}-token prompt at a time, host ids -> first token event); "
                         f"ttft_stage_chain_ms = the same prompt through raw stage.forward + send/recv",
            "ttft_stage_chain_ms": round(ttft_p50 * 1e3, 3),
            "ttft_microbatch_ms": round(ttft_batch * 1e3, 2),
            "clocks": clocks.summary(),
            "gpu_launches": int(launches),
            "e2e": e2e,
        }
        if args.layers:
            res["invalid"] = "truncated model (--layers) — debug run"
        if p2p_err:
            res["invalid"] = "P2P flag wait timed out"
        return res
    return None


def run_ep(args, world, rank, local, dev):
    """Data-parallel attention + expert-parallel MoE: rank r decodes its own ``--batch`` sequences through all layers;
    each MoE layer keeps E/world routed experts per rank and exchanges tokens with the fused dispatch / return kernels
    (``ops/csrc/ep.cu``).  Weights per rank: attention + shared experts + embeddings replicated, routed experts 1/world."""
    import torch
    import torch.distributed as dist

    from mlx_sharding_b200.config import ModelConfig
    from mlx_sharding_b200.engine.core import LLMEngine
    from mlx_sharding_b200.engine.sampler import SamplingParams
    from mlx_sharding_b200.ops import b200
    from mlx_sharding_b200.ops.meta import BatchMeta
    from mlx_sharding_b200.parallel.decode_loop import DecodeLoop
    from mlx_sharding_b200.parallel.ep import enable_expert_parallel
    from mlx_sharding_b200.parallel.pipeline import LocalPipeline, StageExecutor
    from mlx_sharding_b200.utils.loader import random_model
    from mlx_sharding_b200.utils.timing import ClockSampler, max_over_ranks

    log = lambda *a: print(f"[rank {rank}]", *a, file=sys.stderr, flush=True)
    cfgd = model_config(args.model, args.layers)
    cfg = ModelConfig.from_dict(cfgd)
    B, S, PS = args.batch, args.prompt_len, args.page_size
    chunk_seqs = max(1, 2048 // S)                      # prefill chunk: <= 2048 tokens per rank per step
    ep_tokens = max(B, chunk_seqs * S)
    t0 = time.time()
    # same seed on every rank; of every routed-expert bank only this rank's E/world slice is kept as it is generated
    model = random_model(cfgd, dtype=torch.bfloat16, device=dev, backend="b200", seed=1, expert_shard=(rank, world))
    bufs = enable_expert_parallel(model, max_tokens=ep_tokens)
    torch.cuda.synchronize()
    log(f"all {cfg.num_hidden_layers} layers, experts {rank * cfg.n_routed_experts // world}..{(rank + 1) * cfg.n_routed_experts // world - 1} "
        f"of every MoE layer, replicated weights {model.weight_bytes() / 1e9:.2f} GB + expert shards "
        f"{sum(e.wg.numel() + e.wu.numel() + e.wd.numel() for e in model.ep_layers.values()) * 2 / 1e9:.2f} GB built in {time.time() - t0:.1f}s")
    total_steps = args.warmup + args.steps
    e2e_steps = 0 if args.no_e2e else (total_steps + 2)
    max_len = S + total_steps + e2e_steps + 8
    pages_per_seq = (max_len + PS - 1) // PS
    num_pages = B * pages_per_seq * (1 if args.no_e2e else 2) + 1
    stage = StageExecutor(model, num_pages, PS, seed=rank)
    gen = torch.Generator().manual_seed(1234 + rank)
    prompts = torch.randint(3, cfg.vocab_size - 1, (B, S), generator=gen).pin_memory()
    bts = [[1 + b * pages_per_seq + i for i in range(pages_per_seq)] for b in range(B)]

    def prefill(a, b):
        """Prompt ids (pinned host) of sequences [a, b) -> first sampled tokens; all ranks call this in lockstep."""
        meta = BatchMeta.build([S] * (b - a), [0] * (b - a), bts[a:b], PS, device=dev)
        x = prompts[a:b].reshape(-1).to(dev, non_blocking=True)
        return stage.forward(x, meta).argmax(-1)

    def timed(fn):
        dist.barrier()
        torch.cuda.synchronize()
        tt = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return out, time.perf_counter() - tt

    first, batch_ttfts, ttfts = None, [], []
    for rep in range(3):
        parts, dt = timed(lambda: [prefill(a, min(a + chunk_seqs, B)) for a in range(0, B, chunk_seqs)])
        first = torch.cat(parts)
        if rep:
            batch_ttfts.append(dt)
    for rep in range(8):
        _, dt = timed(lambda: prefill(0, 1))
        if rep > 1:
            ttfts.append(dt)
    ttft_p50 = max_over_ranks(statistics.median(ttfts))
    ttft_batch = max_over_ranks(statistics.median(batch_ttfts))
    log(f"prefill done: TTFT p50 {ttft_p50 * 1e3:.2f} ms (1x{S} prompt per rank, all ranks at once), {ttft_batch * 1e3:.1f} ms for {B}x{S} per rank")

    loop = DecodeLoop(stage, 1, B, pages_per_seq, transport="local", use_graphs=not args.no_graphs, standalone=True)
    loop.groups[0].load(torch.full((B,), S, dtype=torch.int32), torch.tensor(bts, dtype=torch.int32), first, max_ctx=max_len)
    loop.capture()
    dist.barrier()
    C = b200.C()
    for _ in range(args.warmup):
        loop.step_all()
    torch.cuda.synchronize()
    dist.barrier()
    n_launch0 = C.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clocks:
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.steps):
            loop.step_all()
        e1.record()
        torch.cuda.synchronize()
    dist.barrier()
    ms = max_over_ranks(e0.elapsed_time(e1))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, decode_outputs(loop, prefix=f"ep_rank{rank}_"), world)
    launches = (loop.launches_per_step * args.steps) if loop.use_graphs else (C.launch_count() - n_launch0)
    ms_per_step = ms / args.steps
    tok_s = world * B * 1000.0 / ms_per_step
    ep_err = bufs.error()
    log(f"decode: {ms_per_step:.3f} ms/step -> {tok_s:.0f} tok/s  (launches/step/rank {launches / max(args.steps, 1):.0f}, ep_err={ep_err})")

    e2e = None
    if not args.no_e2e:
        try:
            # every rank drives its own LLMEngine over the same request shapes, so the engines step in lockstep
            pipe = LocalPipeline([stage])
            eng = LLMEngine(pipe, num_pages, PS, num_groups=1, max_seqs_per_group=B, max_prefill_tokens=chunk_seqs * S)
            n_new = total_steps + 1
            reqs = [eng.submit(prompts[b].tolist(), SamplingParams(temperature=0.0), max_tokens=n_new) for b in range(B)]
            while any(r.prefilled < len(r.prompt) for r in reqs) or min(len(r.output) for r in reqs) < args.warmup:
                eng.step()
            torch.cuda.synchronize()
            dist.barrier()
            h2d0, d2h0 = pipe.h2d_bytes, pipe.d2h_bytes
            n0 = sum(len(r.output) for r in reqs)
            tt = time.perf_counter()
            steps = 0
            while min(len(r.output) for r in reqs) < total_steps:
                eng.step()
                steps += 1
            torch.cuda.synchronize()
            dt = max_over_ranks(time.perf_counter() - tt)
            n1 = sum(len(r.output) for r in reqs)
            eng.drain()
            steps = max(steps, 1)
            h2d1, d2h1 = pipe.h2d_bytes, pipe.d2h_bytes
            ttft = max_over_ranks(engine_ttft(eng, [prompts[(7 * i) % B].tolist() for i in range(TTFT_REQUESTS)]))
            e2e = {"value": round(world * (n1 - n0) / dt, 1), "unit": "tokens/s", "steps": steps, "ms_per_step": round(dt * 1e3 / steps, 4),
                   "h2d_bytes_per_step": int(world * (h2d1 - h2d0) / steps),
                   "d2h_bytes_per_step": int(world * (d2h1 - d2h0) / steps),
                   "ttft_p50_ms": ttft, "ttft_requests": TTFT_REQUESTS,
                   "path": "one LLMEngine.submit/step per rank -> LocalPipeline (pinned H2D of token ids + step metadata, D2H of sampled ids); "
                           "wall time = max over ranks, bytes summed over ranks"}
        except Exception as e:  # noqa: BLE001 — (symmetric) failure of the engine path: keep the device-timed result
            import traceback

            traceback.print_exc()
            e2e = {"error": f"{type(e).__name__}: {e}"}

    dist.barrier()
    if rank == 0:
        res = {
            "metric": METRIC,
            "value": round(tok_s, 1), "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic prompts, random-init weights (mlx-community layout)", "impl": args.impl,
            "config": {"model": "DeepSeek-Coder-V2-Lite-Instruct" if args.model == "deepseek-v2-lite" else args.model,
                       "global_batch": world * B, "seq_len": S, "parallelism": f"ep{world}+dp{world}",
                       "tokens_per_step": world * B, "transport": "fused all-to-all over NVLink peer memory (ops/csrc/ep.cu)",
                       "cuda_graphs": loop.use_graphs, "kv_page_size": PS, "weights": "bf16",
                       "l2": "weights streamed per step far exceed the 126 MB L2; no explicit flush"},
            "ttft_p50_ms": (e2e or {}).get("ttft_p50_ms") or round(ttft_p50 * 1e3, 3),
            "ttft_note": f"p50 over {TTFT_REQUESTS} requests per rank through LLMEngine.submit (one {S}-token prompt at a time, all ranks in lockstep); "
                         f"ttft_stage_chain_ms = raw stage.forward",
            "ttft_stage_chain_ms": round(ttft_p50 * 1e3, 3),
            "ttft_microbatch_ms": round(ttft_batch * 1e3, 2),
            "clocks": clocks.summary(), "gpu_launches": int(launches) * world, "e2e": e2e,
        }
        if args.layers:
            res["invalid"] = "truncated model (--layers) — debug run"
        if ep_err:
            res["invalid"] = "EP flag wait timed out"
        return res
    return None


TTFT_REQUESTS = 32


def engine_ttft(eng, prompt_list):
    """p50 time-to-first-token through the product's public API: one request at a time, ``LLMEngine.submit`` -> first ``TokenEvent``
    (prompt ids start on the host; includes scheduling, the pinned H2D copy, every stage and the D2H of the sampled id)."""
    from mlx_sharding_b200.engine.sampler import SamplingParams

    out = []
    for i, p in enumerate(prompt_list):
        r = eng.submit(p, SamplingParams(temperature=0.0), max_tokens=1)
        while not r.finished:
            eng.step()
        if r.error is not None:
            raise RuntimeError(f"TTFT request failed: {r.error!r}")
        if i >= 2:                      # the first two warm the eager prefill path of this shape
            out.append(r.ttft)
    return round(statistics.median(out) * 1e3, 3)


def run_e2e(args, stage, world, rank, dev, cfg, prompts, G, B, S, num_pages, PS):
    """Same workload through ``LLMEngine`` (the call a user of the serving stack makes)."""
    import torch
    import torch.distributed as dist

    from mlx_sharding_b200.engine.core import LLMEngine
    from mlx_sharding_b200.engine.sampler import SamplingParams
    from mlx_sharding_b200.parallel.pipeline import ChainPipeline, LocalPipeline, worker_loop
    from mlx_sharding_b200.utils.timing import max_over_ranks

    # fresh KV space: pages of the device-timed phase are simply reused (engine has its own allocator)
    if world > 1:
        from mlx_sharding_b200.parallel.pipeline import build_chain

        # the serving chain: shared-memory launch ring + (default) fused P2P hand-off, one CUDA-graph replay per stage per step
        ctl, plane = build_chain(stage, num_groups=G, max_tokens=B * S, max_seqs=B,
                                 transport="auto" if args.transport == "auto" else args.transport)
        if rank != 0:
            worker_loop(stage, ctl, plane)
            return None
        pipe = ChainPipeline(stage, ctl, plane)
    else:
        pipe = LocalPipeline([stage])
    eng = LLMEngine(pipe, num_pages, PS, num_groups=G, max_seqs_per_group=B, max_prefill_tokens=B * S)
    try:
        n_new = args.warmup + args.steps + 1
        reqs = [eng.submit(prompts[g, b].tolist(), SamplingParams(temperature=0.0), max_tokens=n_new)
                for g in range(G) for b in range(B)]

        def failed():
            bad = [r for r in reqs if r.error is not None]
            if bad:
                raise RuntimeError(f"{len(bad)} request(s) failed: {bad[0].error!r}")

        # prefill + warm-up decode steps (untimed)
        while any(r.prefilled < len(r.prompt) for r in reqs) or min(len(r.output) for r in reqs) < args.warmup:
            eng.step()
            failed()
        torch.cuda.synchronize()
        h2d0, d2h0 = pipe.h2d_bytes, pipe.d2h_bytes
        n0 = sum(len(r.output) for r in reqs)
        t0 = time.perf_counter()
        steps = 0
        while min(len(r.output) for r in reqs) < args.warmup + args.steps:
            eng.step()
            steps += 1
            failed()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        n1 = sum(len(r.output) for r in reqs)
        eng.drain()
        steps = max(steps, 1)
        h2d1, d2h1 = pipe.h2d_bytes, pipe.d2h_bytes
        ttft = engine_ttft(eng, [prompts[i % G, (7 * i) % B].tolist() for i in range(TTFT_REQUESTS)])
        return {"value": round((n1 - n0) / dt, 1), "unit": "tokens/s", "steps": steps,
                "ms_per_step": round(dt * 1e3 / steps, 4),
                "h2d_bytes_per_step": int((h2d1 - h2d0) / steps), "d2h_bytes_per_step": int((d2h1 - d2h0) / steps),
                "ttft_p50_ms": ttft, "ttft_requests": TTFT_REQUESTS,
                "path": "LLMEngine.submit/step -> " + type(pipe).__name__ + (f" [{pipe.plane.name} hand-off, {type(pipe.ctl).__name__}]" if world > 1 else "")
                        + " (per step: pinned H2D of the step block = token ids + metadata + sampling block on every stage, D2H of the result message on stage 0)",
                "graph_replays": pipe.gcache.replays if pipe.gcache is not None else 0}
    except Exception as e:  # noqa: BLE001 — the device-timed numbers of this run are still reported
        import traceback

        traceback.print_exc()
        return {"error": f"{type(e).__name__}: {e}"}
    finally:
        if world > 1:
            pipe.shutdown()   # always release the stage workers of the other ranks


if __name__ == "__main__":
    sys.exit(main())
