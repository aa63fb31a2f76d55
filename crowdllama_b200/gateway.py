"""Gateway stand-in: the reference's Ollama-compatible HTTP façade, restated for the benchmark harness.

Mirrors pkg/gateway/gateway.go: POST /api/chat (handleChat :168-231 → FindBestWorker :191 → RequestInference
:243-293) and GET /api/health (:453-461).  SURVEY.md §8f rows 3-4 on top: POST /api/generate (BASELINE.json names
it, the reference gateway lacks it, gateway.go:87-88), the Ollama `options` object passed through to the worker
(GenerateRequest.options), and `"stream": true` answered as NDJSON lines (one per worker frame); Ollama's top-level
`logprobs` / `top_logprobs` travel as options 9 / 10 and come back per token in GenerateResponse.logprobs (`logprobs_json`).  Worker discovery (DHT provider lookup + metadata fetch,
internal/discovery/discovery.go:278-366) is replaced by a static address list whose metadata is polled
over the metadata protocol — the routing rule itself (peermanager FindBestWorker) is `router.find_best_worker`.
Quirks kept: only messages[0].content is forwarded (gateway.go:209); handler errors arrive as assistant
text with HTTP 200 (peer.go:232-243); no worker → 503 JSON error (gateway.go:192-199).
"""
from __future__ import annotations

import json
import random
import socket
import threading
import time
from datetime import datetime, timezone
from http.server import BaseHTTPRequestHandler, ThreadingHTTPServer

from . import handler as H
from .pbwire import read_length_prefixed_pb, write_length_prefixed_pb
from .router import Resource, find_best_worker
from .worker import INFERENCE_PROTOCOL, METADATA_PROTOCOL, _Stream

MAX_TOP_LOGPROBS = 20     # include/clengine.h CL_MAX_TOP_LOGPROBS


def logprobs_json(entries) -> list:
    """GenerateResponse.logprobs (pb.TokenLogprob) -> the reply's "logprobs" array, the shape of Ollama's API
    documentation: one object per generated token with its text, log-probability, UTF-8 bytes and alternatives."""
    def one(t):
        return {"token": t.token.decode("utf-8", "replace"), "logprob": t.logprob, "bytes": list(t.token)}
    return [{**one(t), "top_logprobs": [one(a) for a in t.top_logprobs]} for t in entries]


class PeerTable:
    """peermanager stand-in: address -> Resource, refreshed by metadata probes."""

    def __init__(self, addrs, refresh_s: float = 2.0, seed: int = 0):
        self.addrs = list(addrs)
        self.peers: dict[tuple, Resource] = {}
        self.rng = random.Random(seed)
        self.lock = threading.Lock()
        self.refresh_s = refresh_s
        self._stop = threading.Event()

    def probe(self):
        for a in self.addrs:
            try:
                with socket.create_connection(a, timeout=2) as s:
                    s.sendall((METADATA_PROTOCOL + "\n").encode())
                    data = b""
                    while chunk := s.recv(65536):
                        data += chunk
                r = Resource.from_json(data)
                with self.lock:
                    self.peers[a] = r
            except Exception:  # noqa: BLE001 — refused, reset, closed without JSON, partial JSON: drop THIS peer, keep probing
                with self.lock:
                    self.peers.pop(a, None)

    def start(self):
        self.probe()
        threading.Thread(target=self._loop, daemon=True).start()

    def _loop(self):
        while not self._stop.wait(self.refresh_s):
            self.probe()

    def stop(self):
        self._stop.set()

    def best(self, model: str):
        with self.lock:
            by_id = {r.peer_id: a for a, r in self.peers.items()}
            w = find_best_worker(list(self.peers.values()), model, self.rng)
        return (by_id[w.peer_id], w) if w else (None, None)


def request_inference(addr, model: str, prompt: str, stream: bool, options=None, on_frame=None):
    """Gateway.RequestInference (gateway.go:243-293) over the TCP stand-in for a libp2p stream.  With stream=True the
    worker answers with several frames; on_frame sees each one and the last (Done=true) is returned."""
    with socket.create_connection(addr, timeout=600) as s:
        s.sendall((INFERENCE_PROTOCOL + "\n").encode())
        st = _Stream(s)
        write_length_prefixed_pb(st, H.create_generate_request(model, prompt, stream, options))
        while True:
            g = H.extract_generate_response(read_length_prefixed_pb(st))
            if on_frame is not None:
                on_frame(g)
            if g.done or not stream:
                return g


class _Handler(BaseHTTPRequestHandler):
    protocol_version = "HTTP/1.1"

    def log_message(self, *a):
        pass

    def _json(self, code, obj):
        body = json.dumps(obj).encode()
        self.send_response(code)
        self.send_header("Content-Type", "application/json")
        self.send_header("Content-Length", str(len(body)))
        self.end_headers()
        self.wfile.write(body)

    def do_GET(self):
        if self.path == "/api/health":
            t: PeerTable = self.server.table
            with t.lock:
                peers = {r.peer_id: {"supported_models": r.supported_models, "tokens_throughput": r.tokens_throughput, "load": r.load,
                                     "gpu_model": r.gpu_model} for r in t.peers.values()}
            return self._json(200, {"status": "ok", "peers": peers})
        self._json(404, {"error": "not found"})

    def _ndjson_start(self):
        self.send_response(200)
        self.send_header("Content-Type", "application/x-ndjson")
        self.send_header("Transfer-Encoding", "chunked")
        self.end_headers()

    def _ndjson_line(self, obj):
        body = json.dumps(obj).encode() + b"\n"
        self.wfile.write(f"{len(body):x}\r\n".encode() + body + b"\r\n")
        self.wfile.flush()

    def do_POST(self):
        chat = self.path == "/api/chat"
        if not chat and self.path != "/api/generate":
            return self._json(404, {"error": "not found"})
        try:
            req = json.loads(self.rfile.read(int(self.headers.get("Content-Length", "0"))))
        except Exception:
            return self._json(400, {"error": "invalid JSON"})
        model = req.get("model")
        if chat:
            messages = req.get("messages") or []
            if not model or not messages:                                 # gateway.go:175-188
                return self._json(400, {"error": "model and messages are required"})
            prompt = messages[0].get("content", "")                       # gateway.go:209: only the first message travels
        else:
            prompt = req.get("prompt")
            if not model or prompt is None:
                return self._json(400, {"error": "model and prompt are required"})
        from .pb import GenerateOptions
        options = GenerateOptions.from_json(req.get("options"))
        if not chat and req.get("raw"):
            options = options or GenerateOptions()
            options.raw = True
        want_logprobs = bool(req.get("logprobs", False))
        top_logprobs = req.get("top_logprobs", 0)
        if isinstance(top_logprobs, bool) or not isinstance(top_logprobs, int) or not 0 <= top_logprobs <= MAX_TOP_LOGPROBS:
            return self._json(400, {"error": f"top_logprobs must be an integer within 0..{MAX_TOP_LOGPROBS}"})
        if want_logprobs:
            options = options or GenerateOptions()
            options.logprobs, options.top_logprobs = True, top_logprobs
        stream = bool(req.get("stream", False))
        addr, worker = self.server.table.best(model)
        if worker is None:                                                # gateway.go:192-199
            return self._json(503, {"error": f"no available worker for model {model}"})
        with self.server.lock:
            self.server.counts[worker.peer_id] = self.server.counts.get(worker.peer_id, 0) + 1

        def shape(g):
            now = datetime.now(timezone.utc).isoformat()
            if chat:
                o = {"model": g.model or model, "created_at": now, "message": {"role": "assistant", "content": g.response},
                     "done": g.done}
            else:
                o = {"model": g.model or model, "created_at": now, "response": g.response, "done": g.done}
            if want_logprobs:
                o["logprobs"] = logprobs_json(g.logprobs)
            if g.done:
                o["done_reason"] = g.done_reason
            return o

        if stream:
            started = [False]

            def on_frame(g):
                if not started[0]:
                    self._ndjson_start()
                    started[0] = True
                self._ndjson_line(shape(g))

            try:
                request_inference(addr, model, prompt, True, options, on_frame)
            except Exception as ex:
                if not started[0]:
                    return self._json(500, {"error": f"inference request failed: {ex}"})
                self._ndjson_line({"error": f"inference request failed: {ex}", "done": True})
            self.wfile.write(b"0\r\n\r\n")
            return
        try:
            g = request_inference(addr, model, prompt, False, options)
        except Exception as ex:                                           # gateway.go:210-217
            return self._json(500, {"error": f"inference request failed: {ex}"})
        o = shape(g)
        o["stream"] = False
        o.setdefault("done_reason", g.done_reason)
        self._json(200, o)


class _Server(ThreadingHTTPServer):
    daemon_threads = True
    request_queue_size = 256        # listen() backlog: must be a class attribute, the constructor already listens


def make_server(worker_addrs, port: int = 9001, host: str = "127.0.0.1", seed: int = 0) -> ThreadingHTTPServer:
    srv = _Server((host, port), _Handler)
    srv.table = PeerTable(worker_addrs, seed=seed)
    srv.counts, srv.lock = {}, threading.Lock()
    srv.table.start()
    return srv


def main():
    """python -m crowdllama_b200.gateway --port 9001 --worker 127.0.0.1:9101 --worker 127.0.0.1:9102 ..."""
    import argparse
    ap = argparse.ArgumentParser(description="Ollama-compatible gateway stand-in in front of B200 worker peers")
    ap.add_argument("--host", default="127.0.0.1")
    ap.add_argument("--port", type=int, default=9001)                      # the reference gateway's default port
    ap.add_argument("--worker", action="append", default=[], help="host:port of a worker peer (repeatable)")
    ap.add_argument("--seed", type=int, default=0, help="seed of the random tie-break in FindBestWorker")
    a = ap.parse_args()
    addrs = []
    for w in a.worker or ["127.0.0.1:9101"]:
        h, _, p = w.rpartition(":")
        addrs.append((h or "127.0.0.1", int(p)))
    srv = make_server(addrs, port=a.port, host=a.host, seed=a.seed)
    print(f"gateway on http://{a.host}:{a.port} -> workers {addrs}", flush=True)
    try:
        srv.serve_forever(poll_interval=0.2)
    finally:
        srv.server_close()


if __name__ == "__main__":
    main()
