"""CLI entry points with the reference's flag spellings: generate.py (single process, gRPC peers, torchrun chain),
mlx-sharding-server (ephemeral port print), console-script shims."""
import os
import re
import signal
import subprocess
import sys
import time

import pytest
import torch

from helpers import TINY_LLAMA
from mlx_sharding_b200.utils.checkpoint import write_synthetic_checkpoint

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENV = dict(os.environ, PYTHONPATH=REPO, OMP_NUM_THREADS="1")


@pytest.fixture(scope="module")
def ckpt(tmp_path_factory):
    d = tmp_path_factory.mktemp("cli")
    return write_synthetic_checkpoint(str(d / "tiny"), TINY_LLAMA, dtype=torch.float32)


def _gen(args, timeout=240):
    r = subprocess.run([sys.executable, os.path.join(REPO, "generate.py"), *args], capture_output=True, text=True,
                       env=ENV, timeout=timeout)
    assert r.returncode == 0, r.stdout + r.stderr
    return r.stdout


@pytest.mark.timeout(600)
def test_generate_single_grpc_and_torchrun_agree(ckpt):
    base = ["--model", ckpt, "--prompt", "hello", "--max_tokens", "12", "--device", "cpu"]
    solo = _gen(base)
    assert "Prompt:" in solo and "Generation:" in solo and "tokens-per-sec" in solo
    text = solo.split("=" * 10)[0]
    # reference-style: second stage is an mlx-sharding-server reached over gRPC (ephemeral port printed at start-up)
    srv = subprocess.Popen([sys.executable, "-m", "shard.main", "--model", ckpt, "--start-layer", "2", "--end-layer", "4",
                            "--device", "cpu", "--wire-dtype", "float32"], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                           text=True, env=ENV, start_new_session=True)
    try:
        port, t0 = None, time.time()
        while port is None and time.time() - t0 < 120:
            line = srv.stdout.readline()
            m = re.search(r"listening on port (\d+)", line or "")
            if m:
                port = int(m.group(1))
        assert port, "server did not print its port"
        relay = _gen(base + ["--start_layer", "0", "--end_layer", "2", "--server_address", f"localhost:{port}"])
        assert relay.split("=" * 10)[0] == text
    finally:
        os.killpg(srv.pid, signal.SIGTERM)
    # native chain: torchrun, 2 processes, gloo
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29611", os.path.join(REPO, "generate.py"), *base],
                       capture_output=True, text=True, env=ENV, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.split("=" * 10)[0].strip() == text.strip()


@pytest.mark.timeout(400)
def test_generate_expert_parallel_cpu(tmp_path):
    """``torchrun generate.py --expert_parallel`` on CPU (gloo all_to_all path of parallel/ep.py): experts sharded at load,
    same greedy text as the single-process run."""
    from helpers import TINY_DSV2

    ck = write_synthetic_checkpoint(str(tmp_path / "dsv2"), TINY_DSV2, dtype=torch.float32, seed=4)
    base = ["--model", ck, "--prompt", "experts", "--max_tokens", "10", "--device", "cpu", "--no_chat_template"]
    text = _gen(base).split("=" * 10)[0]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29612", os.path.join(REPO, "generate.py"), *base, "--expert_parallel"],
                       capture_output=True, text=True, env=ENV, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert r.stdout.split("=" * 10)[0] == text and len(text) > 0 and "Generation:" in r.stdout


def test_console_script_targets_exist():
    import shard.main
    import shard.openai_api
    import shard.utils

    assert callable(shard.main.main) and callable(shard.openai_api.main) and callable(shard.utils.load_model)
    p = shard.openai_api.main.__module__
    assert p.endswith("openai_api")
    from mlx_sharding_b200.server.openai_api import build_arg_parser

    a = build_arg_parser().parse_args(["--model", "x", "-s", "h:1,h:2", "-sl", "0", "-el", "14", "--adapter-path", "y",
                                       "--cache-limit-gb", "4", "--use-default-chat-template", "--trust-remote-code",
                                       "--chat-template", "t", "--log-level", "DEBUG", "--static-dir", "z"])
    assert a.llm_shard_addresses == "h:1,h:2" and a.start_layer == 0 and a.end_layer == 14 and a.cache_limit_gb == 4


def _bench_module():
    import importlib.util

    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(REPO, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_result_merge_and_reference_arm(capsys):
    """bench.py host-side contract pieces that need no GPU: the pp/ep result merge and the reference arm's JSON line."""
    import json

    bench = _bench_module()
    pp = dict(value=60.0, ms_per_step=8.0, config={"parallelism": "pp8"}, ttft_p50_ms=8.0, ttft_microbatch_ms=60.0, e2e=None,
              gpu_launches=1, clocks={}, metric="m")
    ep = dict(pp, value=99.0, config={"parallelism": "ep8+dp8"})
    m = bench.merge_results(pp, ep)
    assert m["value"] == 99.0 and m["also_measured"]["layer-range pipeline (config 3)"]["value"] == 60.0
    m = bench.merge_results(pp, dict(ep, invalid="EP flag wait timed out"))
    assert m["value"] == 60.0 and m["also_measured"]["expert parallel (config 5)"]["invalid"]
    m = bench.merge_results(dict(pp, invalid="x"), dict(ep, value=1.0))
    assert m["value"] == 1.0
    assert bench.merge_results(None, ep) is ep
    assert bench.main(["--impl", "reference"]) == 0
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and "unavailable" in line
    a = bench.parse_args([])
    assert a.gpus == 1 and a.warmup >= 3 and a.parallelism == "auto"


def test_bench_dump_outputs(tmp_path):
    """``bench.py --dump-outputs``: the last decode step's token ids (float64) and fp32 logits as .npy; logits over the size
    budget keep a seeded column subset that is the same from run to run."""
    import numpy as np

    from helpers import TINY_DSV2
    from mlx_sharding_b200.config import ModelConfig
    from mlx_sharding_b200.ops.meta import BatchMeta
    from mlx_sharding_b200.parallel.decode_loop import DecodeLoop
    from mlx_sharding_b200.parallel.pipeline import StageExecutor
    from mlx_sharding_b200.utils.loader import random_model

    bench = _bench_module()
    assert bench.parse_args(["--dump-outputs", str(tmp_path)]).dump_outputs == str(tmp_path)
    with pytest.raises(SystemExit):
        bench.parse_args(["--dump-outputs", str(tmp_path), "--impl", "baseline"])

    cfg = ModelConfig.from_dict(TINY_DSV2)
    B, S, PS, steps = 3, 6, 4, 3
    pps = (S + steps + 2 + PS - 1) // PS
    stage = StageExecutor(random_model(TINY_DSV2, dtype=torch.float32), B * pps + 1, PS)
    prompts = torch.randint(3, cfg.vocab_size - 1, (B, S), generator=torch.Generator().manual_seed(3))
    bts = [[1 + b * pps + i for i in range(pps)] for b in range(B)]
    first = stage.forward(prompts.reshape(-1), BatchMeta.build([S] * B, [0] * B, bts, PS)).argmax(-1)
    loop = DecodeLoop(stage, 1, B, pps, use_graphs=False)
    loop.groups[0].load(torch.full((B,), S, dtype=torch.int32), torch.tensor(bts, dtype=torch.int32), first, S + steps + 2)
    loop.capture()
    for _ in range(steps):
        loop.step_all()
    bench.dump_outputs(str(tmp_path / "full"), bench.decode_outputs(loop), 1)
    toks, logits = np.load(tmp_path / "full" / "tokens.npy"), np.load(tmp_path / "full" / "logits.npy")
    assert toks.dtype == np.float64 and toks.shape == (1, B) and logits.dtype == np.float32 and logits.shape == (1, B, cfg.vocab_size)
    assert (toks[0] == logits[0].argmax(-1)).all()           # greedy: the step's sampled ids are its logits' argmax

    bench.DUMP_BYTES = 1_000_000 + 2 * B * 100 * 4           # room for 100 of the 320 vocabulary columns
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"logits": torch.from_numpy(logits)}, 1)
    a, b = np.load(tmp_path / "a" / "logits.npy"), np.load(tmp_path / "b" / "logits.npy")
    assert a.shape == (1, B, 100) and (a == b).all() and set(a[0, 0].tolist()) <= set(logits[0, 0].tolist())
