"""Token log-probabilities without a GPU: the C-ABI symbols and the CL_MAX_TOP_LOGPROBS limit, the missing-device error of
the single-op entry point, the wire extension (GenerateOptions 9 / 10, GenerateResponse 8) and the gateway's JSON
through a mock worker peer."""
import json
import os
import re
import subprocess
import sys
import threading
import urllib.error
import urllib.request
from pathlib import Path

import pytest

from crowdllama_b200 import engine as eng
from crowdllama_b200 import gateway, pb, worker

ROOT = Path(__file__).resolve().parents[1]

_NO_DEVICE_CHILD = r"""
import numpy as np
from crowdllama_b200 import engine as eng
try:
    eng.op_logprobs(np.zeros((2, 300), np.float32), [1, 2], 5)
except eng.EngineError as ex:
    assert ex.status == eng.CL_ERR_NO_DEVICE, ex
else:
    raise SystemExit("cl_op_logprobs ran without a device")
"""


def test_logprobs_symbols_exported_and_declared():
    L = eng.lib()
    header = (ROOT / "include" / "clengine.h").read_text()
    for name in ("cl_op_logprobs", "cl_generate_ids_logprobs", "cl_logprobs_free"):
        assert name in eng.EXPORTS
        assert hasattr(L, name)
        assert re.search(rf"\b{name}\(", header)
    assert re.search(r"typedef struct cl_logprobs \{", header)


def test_max_top_logprobs_matches_header():
    header = (ROOT / "include" / "clengine.h").read_text()
    n = int(re.search(r"#define CL_MAX_TOP_LOGPROBS (\d+)", header).group(1))
    assert n == eng.MAX_TOP_LOGPROBS == gateway.MAX_TOP_LOGPROBS == 20
    # the ABI of the existing structs is unchanged
    assert int(re.search(r"#define CL_ABI_VERSION (\d+)", header).group(1)) == 2
    assert [f for f, _ in eng.Result._fields_][-1] == "n_preempted"


def test_op_logprobs_without_device_returns_no_device():
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHILD], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:] + r.stdout[-2000:]


def _sample_response():
    tops = [pb.TopLogprob(b"Hi", -0.25), pb.TopLogprob(b"\xe2\x82", -1.5), pb.TopLogprob(b"", -3.0)]
    return pb.GenerateResponse(model="m", created_at_seconds=5, response="Hi", done=True, done_reason="stop", worker_id="w",
                               total_duration=9, logprobs=[pb.TokenLogprob(b"Hi", -0.25, tops), pb.TokenLogprob(b"!", 0.0, [])])


def test_pb_round_trips_the_logprob_fields():
    o = pb.GenerateOptions(temperature=0.0, logprobs=True, top_logprobs=7)
    d = pb.GenerateOptions.decode(o.encode())
    assert (d.logprobs, d.top_logprobs, d.temperature, d.raw) == (True, 7, 0.0, None)
    assert pb.GenerateOptions.decode(pb.GenerateOptions(logprobs=False).encode()).logprobs is False   # explicit presence
    fields = [f for f, _, _ in pb._fields(o.encode())]
    assert fields == [2, 9, 10]
    g = _sample_response()
    m = pb.BaseMessage.decode(pb.BaseMessage(generate_response=g).encode()).generate_response
    assert m == g
    assert [t.token for t in m.logprobs[0].top_logprobs] == [b"Hi", b"\xe2\x82", b""]
    assert m.logprobs[1].logprob == 0.0 and m.logprobs[1].top_logprobs == []


def test_pb_old_messages_decode_unchanged():
    """A message without the new fields decodes to empty logprobs; the new fields only append field-8 entries, so a peer
    that does not know field 8 (it skips unknown fields) reads the rest of the frame byte for byte."""
    g = _sample_response()
    old = pb.GenerateResponse(**{k: v for k, v in vars(g).items() if k != "logprobs"})
    assert pb.GenerateResponse.decode(old.encode()).logprobs == []
    new_bytes = g.encode()
    assert new_bytes.startswith(old.encode())
    assert [f for f, _, _ in pb._fields(new_bytes[len(old.encode()):])] == [8, 8]
    r = pb.GenerateRequest(model="m", prompt="p", stream=True, options=pb.GenerateOptions(seed=3, raw=True))
    assert pb.GenerateRequest.decode(r.encode()) == r
    assert pb.GenerateRequest.decode(r.encode()).options.logprobs is None


class _LogprobPeer:
    """Mock engine behind a worker: answers every request with per-token logprob entries (when asked) in one frame, or
    one frame per token when streaming."""
    model_name = "lp"
    words = [b"Hello", b",", b" w\xc3\xb6rld"]

    def stats(self):
        return dict(tokens_per_sec=100.0, load=0.1, vram_gb=179, gpu_model="mock B200")

    def entries(self, opt, words):
        if not (opt and opt.logprobs):
            return []
        k = opt.top_logprobs or 0
        return [pb.TokenLogprob(w, -0.5 * (i + 1), [pb.TopLogprob(w, -0.5 * (i + 1)), pb.TopLogprob(b"x", -2.0)][:k])
                for i, w in enumerate(words)]

    def handler(self):
        def h(ctx, req):
            g = req.generate_request
            self.last = g.options
            return pb.BaseMessage(generate_response=pb.GenerateResponse(
                model=g.model, response=b"".join(self.words).decode(), done=True, done_reason="stop",
                logprobs=self.entries(g.options, self.words)))

        def stream(ctx, req, emit):
            g = req.generate_request
            self.last = g.options
            for w in self.words:
                emit(pb.BaseMessage(generate_response=pb.GenerateResponse(model=g.model, response=w.decode(),
                                                                          logprobs=self.entries(g.options, [w]))))
            emit(pb.BaseMessage(generate_response=pb.GenerateResponse(model=g.model, done=True, done_reason="stop")))
        h.stream = stream
        return h


def _free_port():
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _post(url, obj):
    req = urllib.request.Request(url, json.dumps(obj).encode(), {"Content-Type": "application/json"})
    with urllib.request.urlopen(req, timeout=10) as r:
        body = r.read().decode()
        if r.headers["Content-Type"] == "application/x-ndjson":
            return r.status, [json.loads(x) for x in body.splitlines() if x.strip()]
        return r.status, json.loads(body)


@pytest.fixture
def lp_gateway():
    wp, gp = _free_port(), _free_port()
    peer = _LogprobPeer()
    w = worker.WorkerServer(("127.0.0.1", wp), peer, peer_id="wlp")
    w.api_handler = peer.handler()
    threading.Thread(target=w.serve_forever, daemon=True).start()
    g = gateway.make_server([("127.0.0.1", wp)], port=gp)
    threading.Thread(target=g.serve_forever, daemon=True).start()
    try:
        yield f"http://127.0.0.1:{gp}", peer
    finally:
        g.shutdown(); g.server_close(); w.shutdown(); w.server_close()


def test_gateway_logprobs_json_shape(lp_gateway):
    base, peer = lp_gateway
    st, r = _post(base + "/api/generate", {"model": "lp", "prompt": "x", "logprobs": True, "top_logprobs": 2})
    assert st == 200 and r["response"] == "Hello, wörld" and r["done"]
    assert (peer.last.logprobs, peer.last.top_logprobs) == (True, 2)
    lp = r["logprobs"]
    assert [e["token"] for e in lp] == ["Hello", ",", " wörld"]
    assert lp[2]["bytes"] == list(b" w\xc3\xb6rld") and lp[0]["logprob"] == -0.5
    assert lp[0]["top_logprobs"] == [{"token": "Hello", "logprob": -0.5, "bytes": list(b"Hello")},
                                     {"token": "x", "logprob": -2.0, "bytes": [120]}]
    assert set(lp[1]) == {"token", "logprob", "bytes", "top_logprobs"}
    st, r = _post(base + "/api/chat", {"model": "lp", "messages": [{"role": "user", "content": "x"}], "logprobs": True})
    assert r["message"]["content"] == "Hello, wörld" and len(r["logprobs"]) == 3
    assert all(e["top_logprobs"] == [] for e in r["logprobs"]) and peer.last.top_logprobs == 0


def test_gateway_streams_logprobs_per_frame(lp_gateway):
    base, _ = lp_gateway
    for path, body in (("/api/generate", {"prompt": "x"}), ("/api/chat", {"messages": [{"role": "user", "content": "x"}]})):
        st, lines = _post(base + path, {"model": "lp", "stream": True, "logprobs": True, "top_logprobs": 1, **body})
        assert st == 200 and len(lines) == 4 and lines[-1]["done"] and lines[-1]["logprobs"] == []
        for line, w in zip(lines, _LogprobPeer.words):
            text = line["response"] if path == "/api/generate" else line["message"]["content"]
            assert text == w.decode()
            assert [e["token"] for e in line["logprobs"]] == [w.decode()] and len(line["logprobs"][0]["top_logprobs"]) == 1


def test_gateway_rejects_top_logprobs_out_of_range(lp_gateway):
    base, _ = lp_gateway
    for bad in (21, -1, "5", 2.5):
        with pytest.raises(urllib.error.HTTPError) as ei:
            _post(base + "/api/generate", {"model": "lp", "prompt": "x", "logprobs": True, "top_logprobs": bad})
        assert ei.value.code == 400


def test_gateway_without_logprobs_returns_none(lp_gateway):
    base, peer = lp_gateway
    for extra in ({}, {"logprobs": False}, {"logprobs": False, "top_logprobs": 3}):
        st, r = _post(base + "/api/generate", {"model": "lp", "prompt": "x", **extra})
        assert st == 200 and "logprobs" not in r and not (peer.last and peer.last.logprobs)
        st, lines = _post(base + "/api/chat", {"model": "lp", "stream": True, "messages": [{"role": "user", "content": "x"}], **extra})
        assert all("logprobs" not in x for x in lines)
