"""Multi-process API front end (server/frontend.py): HTTP / SSE / tokenizer in worker processes, engine loop in this one.
The responses must equal the in-process server's for the same greedy requests; errors, cancellation and /metrics cross the
process boundary."""
import http.client
import json
import os
import socket
import threading
import time

import pytest
import torch

from helpers import TINY_LLAMA
from mlx_sharding_b200.server import openai_api
from mlx_sharding_b200.server.frontend import FrontEnd
from mlx_sharding_b200.utils.checkpoint import write_synthetic_checkpoint


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.fixture(scope="module")
def servers(tmp_path_factory):
    d = tmp_path_factory.mktemp("ckpt")
    path = write_synthetic_checkpoint(str(d / "tiny"), TINY_LLAMA, dtype=torch.float32)
    cwd = os.getcwd()
    os.chdir(d)
    # the tiny model's head dim (16) has no sm_100a attention kernel: keep it on the CPU path on a machine with a GPU too
    args = openai_api.build_arg_parser().parse_args(["--model", path, "--port", "0", "--kv-pages", "128", "--page-size", "16",
                                                     "--device", "cpu"])
    args.static_dir = os.path.join(os.path.dirname(openai_api.__file__), "static")
    provider = openai_api.ModelProvider(args, [])
    httpd = openai_api.make_server("127.0.0.1", 0, provider, args.static_dir)          # in-process server: the oracle
    threading.Thread(target=httpd.serve_forever, daemon=True).start()
    port = _free_port()
    front = FrontEnd(provider.engine, 2, "127.0.0.1", port, args.static_dir, path, "default_model", {}, "WARNING").start()
    yield port, httpd.server_address[1], provider
    front.stop()
    httpd.shutdown()
    provider.engine.shutdown()
    os.chdir(cwd)


def _post(port, path, body, raw=False):
    c = http.client.HTTPConnection("127.0.0.1", port, timeout=120)
    c.request("POST", path, json.dumps(body), {"Content-Type": "application/json"})
    r = c.getresponse()
    data = r.read()
    c.close()
    return r, (data if raw else json.loads(data))


def test_completion_matches_in_process_server(servers):
    wport, iport, _ = servers
    body = {"prompt": "hello world", "max_tokens": 9, "temperature": 0, "logprobs": 3}
    rw, jw = _post(wport, "/v1/completions", body)
    ri, ji = _post(iport, "/v1/completions", body)
    assert rw.status == ri.status == 200
    assert jw["choices"][0]["logprobs"]["tokens"] == ji["choices"][0]["logprobs"]["tokens"]
    assert jw["choices"][0]["text"] == ji["choices"][0]["text"] and jw["usage"] == ji["usage"]
    assert jw["choices"][0]["logprobs"]["top_logprobs"] == ji["choices"][0]["logprobs"]["top_logprobs"]


def test_streams_from_many_clients(servers):
    wport, iport, _ = servers
    n = 12
    out = [None] * n

    def one(i):
        body = {"messages": [{"role": "user", "content": f"request {i}"}], "max_tokens": 6 + i % 3, "temperature": 0, "stream": True}
        r, raw = _post(wport, "/v1/chat/completions", body, raw=True)
        ev = [l[6:] for l in raw.decode().split("\n\n") if l.startswith("data: ")]
        text = "".join(json.loads(e)["choices"][0]["delta"]["content"] for e in ev[:-1])
        _, j = _post(iport, "/v1/chat/completions", dict(body, stream=False))
        out[i] = (r.status, ev[-1], text, j["choices"][0]["message"]["content"], json.loads(ev[-2])["choices"][0]["finish_reason"])

    th = [threading.Thread(target=one, args=(i,)) for i in range(n)]
    [t.start() for t in th]
    [t.join() for t in th]
    for status, last, text, want, reason in out:
        assert status == 200 and last == "[DONE]" and text == want and reason in ("length", "stop")


def test_errors_and_zero_tokens_cross_the_process_boundary(servers):
    wport, _, _ = servers
    r, j = _post(wport, "/v1/completions", {"prompt": "x" * 5000, "max_tokens": 100000})      # engine-side validation -> 400
    assert r.status == 400 and "max_model_len" in j["error"]["message"]
    r, j = _post(wport, "/v1/completions", {"prompt": "abc", "max_tokens": 0})
    assert r.status == 200 and j["choices"][0]["text"] == "" and j["usage"]["completion_tokens"] == 0
    r, j = _post(wport, "/v1/completions", {"prompt": "abc", "max_tokens": 2, "model": "some/other"})   # no hot-swap from a worker
    assert r.status == 400 and "cannot be switched" in j["error"]["message"]
    r, j = _post(wport, "/v1/completions", {"prompt": "abc", "temperature": -1})
    assert r.status == 400


def test_metrics_and_client_disconnect(servers):
    wport, _, provider = servers
    c = http.client.HTTPConnection("127.0.0.1", wport, timeout=30)
    c.request("GET", "/metrics")
    text = c.getresponse().read().decode()
    assert "mlx_sharding_engine_steps" in text and "mlx_sharding_kv_pages_free" in text
    free0 = provider.engine.table.alloc.num_free
    # a client that walks away mid-stream: the worker cancels the request in the engine process, pages come back
    s = socket.create_connection(("127.0.0.1", wport))
    body = json.dumps({"prompt": "abc", "max_tokens": 400, "temperature": 0, "stream": True}).encode()
    s.sendall(b"POST /v1/completions HTTP/1.1\r\nHost: x\r\nContent-Type: application/json\r\nContent-Length: %d\r\n\r\n" % len(body) + body)
    s.recv(200)
    s.close()
    for _ in range(300):
        if not provider.engine.busy() and provider.engine.table.alloc.num_free == free0:
            break
        time.sleep(0.05)
    assert not provider.engine.busy() and provider.engine.table.alloc.num_free == free0


def test_stop_sequences_logit_bias_and_seeded_sampling_through_workers(servers):
    """Request features that live on both sides of the pipe: stop sequences (engine stops, handler trims / holds text back),
    logit bias + top-logprobs (sampling block), per-request seeds (same seed -> same tokens, from either front end)."""
    wport, iport, _ = servers
    body = {"prompt": "abc", "max_tokens": 10, "temperature": 0, "logit_bias": {"65": 100.0}, "stop": "AA", "logprobs": 2}
    rw, jw = _post(wport, "/v1/completions", body)
    ri, ji = _post(iport, "/v1/completions", body)
    assert jw["choices"][0]["finish_reason"] == "stop" and jw["choices"][0]["text"] == "" and jw["choices"][0] == ji["choices"][0]
    # streaming with a stop sequence: held-back text never reaches the client
    r, raw = _post(wport, "/v1/completions", dict(body, stream=True), raw=True)
    ev = [json.loads(l[6:]) for l in raw.decode().split("\n\n") if l.startswith("data: ") and l[6:] != "[DONE]"]
    assert "".join(e["choices"][0]["text"] for e in ev) == "" and ev[-1]["choices"][0]["finish_reason"] == "stop"
    # sampled requests: reproducible per seed, identical from a worker and from the in-process server
    samp = {"prompt": "seeded", "max_tokens": 12, "temperature": 1.0, "top_p": 0.9, "seed": 1234}
    a = _post(wport, "/v1/completions", samp)[1]["choices"][0]["logprobs"]["tokens"]
    b = _post(wport, "/v1/completions", samp)[1]["choices"][0]["logprobs"]["tokens"]
    c = _post(iport, "/v1/completions", samp)[1]["choices"][0]["logprobs"]["tokens"]
    d = _post(wport, "/v1/completions", dict(samp, seed=99))[1]["choices"][0]["logprobs"]["tokens"]
    assert a == b == c and len(a) == 12 and d != a


def test_engine_bridge_under_load_without_http():
    """RemoteEngine <-> _WorkerSink over a pipe inside one process, stub pipeline (no model): many concurrent requests with different
    lengths, a few cancelled mid-stream — every stream ends exactly once with the right number of tokens, nothing is left behind."""
    import multiprocessing as mp
    import random

    from mlx_sharding_b200.engine.core import LLMEngine, StepOutput
    from mlx_sharding_b200.engine.sampler import SamplingParams
    from mlx_sharding_b200.server.frontend import RemoteEngine, _WorkerSink

    class Stub:
        num_stages = 2

        def submit(self, inp):
            n = inp.meta.num_seqs
            return StepOutput(tokens=[7] * n, logprobs=[0.0] * n)

        def wait(self, h):
            return h

        def reset(self):
            pass

    eng = LLMEngine(Stub(), 4096, 16, num_groups=2, max_seqs_per_group=16, max_prefill_tokens=256).start()
    free0 = eng.table.alloc.num_free
    a, b = mp.Pipe(duplex=True)
    sink = _WorkerSink(a, eng)
    eng.sinks.append(sink)
    remote = RemoteEngine(b)
    rnd = random.Random(3)
    plan = [(rnd.randint(1, 40), rnd.random() < 0.15) for _ in range(120)]
    results = [None] * len(plan)

    def run(i):
        n, cancel = plan[i]
        r = remote.submit(list(range(3, 3 + rnd.randint(1, 30))), SamplingParams(temperature=0.0), max_tokens=n, eos_token_id=None)
        got, reason = 0, None
        for ev in r:
            if ev.token < 0:
                reason = ev.finish_reason
                break
            got += 1
            if cancel and got == 1:
                r.cancel()
            if ev.finished:
                reason = ev.finish_reason
        results[i] = (got, reason)

    th = [threading.Thread(target=run, args=(i,)) for i in range(len(plan))]
    [t.start() for t in th]
    [t.join(timeout=120) for t in th]
    assert all(not t.is_alive() for t in th)
    for (n, cancel), (got, reason) in zip(plan, results):
        if cancel and n > 2:
            assert reason in ("cancelled", "length") and 1 <= got <= n       # the cancel races with the engine: it may finish first
        else:
            assert got == n and reason == "length"
    for _ in range(100):
        if not eng.busy() and not sink.requests and not remote.reqs:
            break
        time.sleep(0.05)
    assert not eng.busy() and not sink.requests and not remote.reqs
    assert eng.table.alloc.num_free == free0
    eng.shutdown()
    a.close()
    b.close()
