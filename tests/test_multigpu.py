"""Multi-GPU tests (torchrun, one rank per GPU): fused-P2P / NCCL pipeline parity with a single-GPU run, and
expert-parallel MoE parity.  Skipped unless >= 2 CUDA devices are visible."""
import os
import subprocess
import sys

import pytest

pytestmark = [pytest.mark.gpu, pytest.mark.multigpu]
HERE = os.path.dirname(os.path.abspath(__file__))


def _torchrun(script, args, nproc=2, port=29571, timeout=420):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(HERE, "mgpu", script), *args]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout)
    return r.stdout + r.stderr


@pytest.mark.parametrize("arch,transport,port", [("dsv2", "fused", 29571), ("llama", "fused", 29572), ("dsv2", "nccl", 29573),
                                                 ("dsv2", "fused,half", 29575), ("gemma2", "fused", 29579)])
def test_pipeline_parity(arch, transport, port):
    """``fused,half``: the stage boundary sits between the attention and the MLP block (o-proj epilogue does the P2P store)."""
    out = _torchrun("pipeline_parity.py", [arch] + transport.split(","), port=port)
    assert "PARITY_OK" in out, out[-3000:]


@pytest.mark.parametrize("arch,transport,port", [("dsv2", "fused", 29581), ("llama", "fused", 29582), ("dsv2", "nccl", 29583)])
def test_serving_chain_parity(arch, transport, port):
    """The product path: LLMEngine -> ChainPipeline (shared-memory launch ring, fused P2P hand-off inside per-stage CUDA graphs),
    greedy + seeded sampled requests, against a single-GPU engine."""
    out = _torchrun("serving_chain_parity.py", [arch, transport], port=port)
    assert "SERVING_OK" in out, out[-3000:]


# (the "v2" test ids name the expert exchange as it was called when a second one still existed)
@pytest.mark.parametrize("port", [pytest.param(29574, id="v2-29574")])
def test_expert_parallel_moe(port):
    """Sender-side slot reservation + arrival wait fused into the grouped GEMM == the local MoE, eagerly and under graph replay."""
    out = _torchrun("ep_parity.py", [], port=port)
    assert "EP_OK" in out, out[-3000:]


@pytest.mark.parametrize("mode,port", [pytest.param("forward", 29584, id="v2-29584"), ("fused", 29586)])
def test_expert_parallel_stress(mode, port):
    """Several EP layers sharing one buffer set, called back to back with no host synchronisation, token counts changing from step
    to step (prefill chunk <-> decode batch), two geometries; every output must equal the local MoE bit for bit.  ``forward``: rows
    routed separately; ``fused``: the four-kernel block (norm + router + dispatch in one kernel, combine + next norm in one)
    against separate kernels."""
    out = _torchrun("ep_stress.py", [mode], port=port)
    assert "EP_STRESS_OK " + mode in out, out[-3000:]


def test_expert_parallel_whole_model():
    """Data-parallel attention + expert-parallel MoE for every layer, graph-captured decode loop (bench.py --parallelism ep)."""
    out = _torchrun("ep_model_parity.py", [], port=29576)
    assert "EP_MODEL_OK" in out, out[-3000:]


def test_generate_cli_expert_parallel(tmp_path):
    """``torchrun generate.py --expert_parallel`` (experts sharded at load, fused all-to-all) prints the same greedy text as a
    single-GPU run of the whole model."""
    import torch

    sys.path.insert(0, HERE)
    from helpers import GPU_DSV2
    from mlx_sharding_b200.utils.checkpoint import write_synthetic_checkpoint

    ckpt = write_synthetic_checkpoint(str(tmp_path / "dsv2"), GPU_DSV2, dtype=torch.bfloat16, seed=11)
    root = os.path.dirname(HERE)
    common = ["--model", ckpt, "--prompt", "expert parallel", "--max_tokens", "12", "--no_chat_template"]
    one = subprocess.run([sys.executable, os.path.join(root, "generate.py"), *common], capture_output=True, text=True, timeout=300,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES="0"))
    assert one.returncode == 0, one.stderr[-2000:]
    ep = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                         "--master-port", "29577", os.path.join(root, "generate.py"), *common, "--expert_parallel"],
                        capture_output=True, text=True, timeout=420)
    assert ep.returncode == 0, (ep.stdout + ep.stderr)[-3000:]
    # NCCL prints a version banner on stdout when NCCL_DEBUG=VERSION is set in the environment: not part of the generation
    text = lambda out: "".join(l for l in out.split("==========")[0].splitlines(True) if not l.startswith("NCCL version"))
    assert "Generation:" in ep.stdout
    assert text(one.stdout) == text(ep.stdout) and len(text(one.stdout)) > 0


# ---------------------------------------------------------------------------------------------- HTTP serving on GPUs
def _serve_and_ask(tmp_path, ckpt, nproc, extra, bodies, master_port):
    """Start ``mlx-sharding-api`` (plain or under torchrun), POST ``bodies`` concurrently, return (answers, /metrics text)."""
    import concurrent.futures
    import http.client
    import json
    import signal
    import socket
    import time

    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        http_port = s.getsockname()[1]
    root = os.path.dirname(HERE)
    cmd = [sys.executable, "-m", "shard.openai_api"] if nproc == 1 else \
        [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}", "--master-addr", "127.0.0.1",
         "--master-port", str(master_port), "-m", "shard.openai_api"]
    cmd += ["--model", ckpt, "--port", str(http_port), "--kv-pages", "256", "--page-size", "64", "--log-level", "WARNING"] + extra
    env = dict(os.environ, PYTHONPATH=root)
    if nproc == 1:
        env["CUDA_VISIBLE_DEVICES"] = "0"
    log_path = os.path.join(str(tmp_path), f"server_{nproc}_{'_'.join(e.strip('-') for e in extra) or 'plain'}.log")
    log_f = open(log_path, "wb")
    proc = subprocess.Popen(cmd, cwd=str(tmp_path), env=env, stdout=log_f, stderr=subprocess.STDOUT, start_new_session=True)
    tail = lambda: open(log_path, errors="replace").read()[-4000:]

    def post(body):
        c = http.client.HTTPConnection("127.0.0.1", http_port, timeout=180)
        c.request("POST", "/v1/chat/completions", json.dumps(body), {"Content-Type": "application/json"})
        r = c.getresponse()
        data = r.read()
        c.close()
        return r.status, json.loads(data)

    try:
        t0 = time.time()
        while True:
            assert proc.poll() is None, "server exited early: " + tail()
            assert time.time() - t0 < 300, "server did not come up"
            try:
                c = http.client.HTTPConnection("127.0.0.1", http_port, timeout=2)
                c.request("GET", "/health")
                if c.getresponse().status == 200:
                    break
            except OSError:
                time.sleep(0.5)
        try:
            with concurrent.futures.ThreadPoolExecutor(len(bodies)) as ex:
                res = list(ex.map(post, bodies))
        except Exception as e:  # noqa: BLE001 — show what the server printed
            time.sleep(1.0)
            raise AssertionError(f"request failed ({type(e).__name__}: {e}); server log tail:\n" + tail()) from e
        c = http.client.HTTPConnection("127.0.0.1", http_port, timeout=10)
        c.request("GET", "/metrics")
        metrics = c.getresponse().read().decode()
        return res, metrics
    finally:
        os.killpg(proc.pid, signal.SIGTERM)      # the exact process group started above
        try:
            proc.wait(timeout=30)
        except subprocess.TimeoutExpired:
            os.killpg(proc.pid, signal.SIGKILL)
        log_f.close()


def _agree(a, b):
    """Greedy answers of two numerically different executions of the same model: equal lengths, equal first token, and at most one
    request diverging later (a near-tie flips the rest of that stream)."""
    assert [len(x) for x in a] == [len(x) for x in b]
    assert all(x[0] == y[0] for x, y in zip(a, b))
    assert sum(x != y for x, y in zip(a, b)) <= 1, (a, b)


@pytest.mark.timeout(900)
def test_http_serving_on_gpus(tmp_path):
    """``mlx-sharding-api`` on real GPUs, the three layouts a user can start: one GPU; a 2-stage chain under torchrun with the HTTP
    front end in worker processes (``--api-workers``); a 2-rank expert-parallel lockstep group.  Same greedy answers."""
    import torch

    sys.path.insert(0, HERE)
    from helpers import GPU_DSV2
    from mlx_sharding_b200.utils.checkpoint import write_synthetic_checkpoint

    ckpt = write_synthetic_checkpoint(str(tmp_path / "dsv2"), GPU_DSV2, dtype=torch.bfloat16, seed=11)
    bodies = [{"messages": [{"role": "user", "content": f"hello gpus {i}"}], "max_tokens": 6 + i, "temperature": 0, "logprobs": 1}
              for i in range(4)]
    toks = lambda res: [j["choices"][0]["logprobs"]["tokens"] for _, j in res]
    one, _ = _serve_and_ask(tmp_path, ckpt, 1, [], bodies, 0)
    assert all(st == 200 for st, _ in one) and [len(t) for t in toks(one)] == [6, 7, 8, 9]
    chain, m = _serve_and_ask(tmp_path, ckpt, 2, ["--api-workers", "2"], bodies, 29591)
    assert all(st == 200 for st, _ in chain), chain
    _agree(toks(one), toks(chain))
    assert "mlx_sharding_engine_steps" in m
    ep, m = _serve_and_ask(tmp_path, ckpt, 2, ["--expert-parallel"], bodies, 29592)
    assert all(st == 200 for st, _ in ep), ep
    _agree(toks(one), toks(ep))
    assert "lockstep_assigned_rank0 2" in m and "lockstep_assigned_rank1 2" in m, m
