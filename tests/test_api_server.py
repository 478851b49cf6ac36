"""Black-box HTTP tests of the OpenAI-compatible server with a tiny model on the CPU path (SURVEY §4)."""
import http.client
import json
import os
import threading

import pytest
import torch

from helpers import TINY_LLAMA
from mlx_sharding_b200.server import openai_api
from mlx_sharding_b200.utils.checkpoint import write_synthetic_checkpoint


@pytest.fixture(scope="module")
def server(tmp_path_factory):
    d = tmp_path_factory.mktemp("ckpt")
    path = write_synthetic_checkpoint(str(d / "tiny"), TINY_LLAMA, dtype=torch.float32)
    cwd = os.getcwd()
    os.chdir(d)
    # the tiny model's head dim (16) has no sm_100a attention kernel: keep it on the CPU path on a machine with a GPU too
    args = openai_api.build_arg_parser().parse_args(["--model", path, "--port", "0", "--kv-pages", "128", "--page-size", "16", "--prefix-cache",
                                                     "--device", "cpu"])
    args.static_dir = os.path.join(os.path.dirname(openai_api.__file__), "static")
    provider = openai_api.ModelProvider(args, [])
    httpd = openai_api.make_server("127.0.0.1", 0, provider, args.static_dir)
    t = threading.Thread(target=httpd.serve_forever, daemon=True)
    t.start()
    yield httpd.server_address[1], provider
    httpd.shutdown()
    provider.engine.shutdown()
    os.chdir(cwd)


def _post(port, path, body, raw=False):
    c = http.client.HTTPConnection("127.0.0.1", port, timeout=60)
    c.request("POST", path, json.dumps(body), {"Content-Type": "application/json"})
    r = c.getresponse()
    data = r.read()
    c.close()
    return r, (data if raw else json.loads(data))


def test_text_completion_envelope(server):
    port, _ = server
    r, j = _post(port, "/v1/completions", {"prompt": "hello", "max_tokens": 5, "temperature": 0})
    assert r.status == 200 and r.getheader("Access-Control-Allow-Origin") == "*"
    assert j["object"] == "text_completion" and j["id"].startswith("cmpl-") and j["model"] == "default_model"
    ch = j["choices"][0]
    assert ch["index"] == 0 and ch["finish_reason"] in ("length", "stop") and isinstance(ch["text"], str)
    assert j["usage"]["prompt_tokens"] == 5 and j["usage"]["completion_tokens"] == len(ch["logprobs"]["tokens"])
    assert j["usage"]["total_tokens"] == j["usage"]["prompt_tokens"] + j["usage"]["completion_tokens"]
    assert j["system_fingerprint"].startswith("fp_")


def test_chat_completion_and_determinism(server):
    port, _ = server
    body = {"messages": [{"role": "user", "content": "hi there"}], "max_tokens": 6, "temperature": 0}
    r1, j1 = _post(port, "/v1/chat/completions", body)
    r2, j2 = _post(port, "/chat/completions", body)
    assert j1["object"] == "chat.completions" and j1["id"].startswith("chatcmpl-")
    assert j1["choices"][0]["message"]["role"] == "assistant"
    assert j1["choices"][0]["logprobs"]["tokens"] == j2["choices"][0]["logprobs"]["tokens"]


def test_logprobs_and_logit_bias(server):
    port, _ = server
    r, j = _post(port, "/v1/completions", {"prompt": "abc", "max_tokens": 3, "temperature": 0, "logprobs": 4,
                                           "logit_bias": {"65": 100.0}})
    lp = j["choices"][0]["logprobs"]
    assert lp["tokens"] == [65, 65, 65] and j["choices"][0]["text"] == "AAA"
    assert len(lp["top_logprobs"]) == 3 and all(len(d) == 4 for d in lp["top_logprobs"])
    assert all(abs(d["65"] - t) < 1e-4 for d, t in zip(lp["top_logprobs"], lp["token_logprobs"]))


def test_stop_sequence_trims_text(server):
    port, _ = server
    r, j = _post(port, "/v1/completions", {"prompt": "abc", "max_tokens": 10, "temperature": 0,
                                           "logit_bias": {"65": 100.0}, "stop": "AA"})
    assert j["choices"][0]["finish_reason"] == "stop" and j["choices"][0]["text"] == ""
    assert j["choices"][0]["logprobs"]["tokens"] == [65, 65]


def test_streaming_sse(server):
    port, _ = server
    body = {"messages": [{"role": "user", "content": "stream please"}], "max_tokens": 8, "temperature": 0,
            "stream": True, "logit_bias": {"66": 50.0}}
    r, raw = _post(port, "/v1/chat/completions", body, raw=True)
    assert r.status == 200 and r.getheader("Content-type") == "text/event-stream"
    events = [l[6:] for l in raw.decode().split("\n\n") if l.startswith("data: ")]
    assert events[-1] == "[DONE]"
    chunks = [json.loads(e) for e in events[:-1]]
    assert all(c["object"] == "chat.completions.chunk" and "usage" not in c for c in chunks)
    assert all(c["choices"][0]["finish_reason"] is None for c in chunks[:-1])
    assert chunks[-1]["choices"][0]["finish_reason"] == "length"
    text = "".join(c["choices"][0]["delta"]["content"] for c in chunks)
    assert text == "B" * 8  # logit_bias is honoured in streaming mode (the reference drops it)


def test_validation_404_options_static(server):
    port, _ = server
    r, j = _post(port, "/v1/completions", {"prompt": "x", "temperature": -1})
    assert r.status == 400 and "temperature" in j["error"]["message"]
    r, j = _post(port, "/v1/completions", {"prompt": "x", "logprobs": 11})
    assert r.status == 400
    r, j = _post(port, "/v1/chat/completions", {"max_tokens": 1})
    assert r.status == 400
    r, raw = _post(port, "/v1/nope", {}, raw=True)
    assert r.status == 404 and raw == b"Not Found"
    r, raw = _post(port, "/v1/completions", {"prompt": "x", "model": "/definitely/not/here"}, raw=True)
    assert r.status == 404
    c = http.client.HTTPConnection("127.0.0.1", port, timeout=30)
    c.request("OPTIONS", "/v1/chat/completions")
    r = c.getresponse(); r.read()
    assert r.status == 204 and r.getheader("Access-Control-Allow-Methods") == "*"
    c.request("GET", "/")
    r = c.getresponse(); html = r.read()
    assert r.status == 200 and b"<html" in html and r.getheader("Content-type") == "text/html"
    c.request("GET", "/app.js")
    r = c.getresponse(); r.read()
    assert r.status == 200
    c.request("GET", "/../../etc/passwd")
    r = c.getresponse(); r.read()
    assert r.status == 404
    c.request("GET", "/metrics")
    r = c.getresponse(); m = r.read().decode()
    assert "mlx_sharding_requests" in m
    c.close()


def test_concurrent_requests(server):
    port, _ = server
    outs = {}

    def go(i):
        outs[i] = _post(port, "/v1/completions", {"prompt": "same prompt", "max_tokens": 6, "temperature": 0})[1]

    ts = [threading.Thread(target=go, args=(i,)) for i in range(6)]
    [t.start() for t in ts]
    [t.join(60) for t in ts]
    toks = [outs[i]["choices"][0]["logprobs"]["tokens"] for i in range(6)]
    assert all(t == toks[0] for t in toks)


def test_convert_chat_fallback():
    s = openai_api.convert_chat([{"role": "system", "content": "be nice"}, {"role": "user", "content": "hi"}])
    assert s == "ASSISTANT's RULE: be nice\nUSER: hi\nASSISTANT:"


def test_prefix_cache_hits_show_up_in_metrics(server):
    """The server fixture runs with --prefix-cache: repeating a long prompt re-uses its KV pages and answers identically."""
    port, provider = server
    body = {"prompt": "the quick brown fox jumps over the lazy dog " * 3, "max_tokens": 6, "temperature": 0}
    _, a = _post(port, "/v1/completions", body)
    before = provider.engine.stats["prefix_cached_tokens"]
    _, b = _post(port, "/v1/completions", body)
    assert a["choices"][0]["text"] == b["choices"][0]["text"]
    assert provider.engine.stats["prefix_cached_tokens"] > before
    c = http.client.HTTPConnection("127.0.0.1", port, timeout=10)
    c.request("GET", "/metrics")
    assert "mlx_sharding_engine_prefix_cached_tokens" in c.getresponse().read().decode()
