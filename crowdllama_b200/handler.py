"""Host-side mirror of the reference's handler interface for the hot path.

  UnifiedAPIHandler        /root/reference/pkg/crowdllama/api.go:19
  WorkerAPIHandler         api.go:45-96   -> worker_api_handler(engine): the B200 engine behind the
                                             same closure shape (the Go cgo shim in go/b200handler
                                             does exactly this around cl_generate)
  DefaultAPIHandler        api.go:163-189 -> default_api_handler (consumer echo)
  CreateGenerateRequest /
  Extract*                 api.go:192-222
  handleInferenceRequest   /root/reference/pkg/peer/peer.go:190-256 -> handle_inference_stream

The Go toolchain is absent from this image, so this module is what the parity / envelope tests and
the multi-worker benchmark harness drive; names, argument meaning and error behaviour follow the
reference so the tests read like pkg/ipc/ipc_test.go and test/integration_test.go.
"""
from __future__ import annotations

import time
from typing import Callable

from . import engine as eng
from .pb import BaseMessage, GenerateRequest, GenerateResponse
from .pbwire import read_length_prefixed_pb, write_length_prefixed_pb

UnifiedAPIHandler = Callable[[object, BaseMessage], BaseMessage]


class HandlerError(Exception):
    pass


def merge_sampling(base: "eng.Sampling | None", options) -> "eng.Sampling | None":
    """Request options (pb.GenerateOptions, the §8f-row-3 wire extension) override the worker's default sampling
    field by field — the same rule as apply_options() inside libclengine (csrc/host_util.cpp)."""
    if options is None or options.is_empty():
        return base
    s = eng.Sampling()
    if base is not None:
        for name, _ in eng.Sampling._fields_:
            setattr(s, name, getattr(base, name))
    else:
        d = eng.ollama_default_sampling(seed=time.time_ns() & 0xFFFFFFFF)
        for name, _ in eng.Sampling._fields_:
            setattr(s, name, getattr(d, name))
    for src, dst in (("seed", "seed"), ("temperature", "temperature"), ("top_k", "top_k"), ("top_p", "top_p"),
                     ("repeat_penalty", "repeat_penalty"), ("repeat_last_n", "repeat_last_n"), ("num_predict", "max_new_tokens")):
        v = getattr(options, src)
        if v is not None:
            setattr(s, dst, v)
    return s


def _response(model: str, text: str, done: bool, done_reason: str = "") -> BaseMessage:
    now = time.time_ns()
    return BaseMessage(generate_response=GenerateResponse(
        model=model, created_at_seconds=now // 10**9, created_at_nanos=now % 10**9, response=text, done=done,
        done_reason=done_reason,
        worker_id="worker",                                          # api.go:83 (literal)
        total_duration=now if done else 0))                          # api.go:84 (absolute UnixNano in the reference)


def worker_api_handler(engine: "eng.Engine", sampling: "eng.Sampling | None" = None) -> UnifiedAPIHandler:
    """WorkerAPIHandler(ollamaBaseURL) with the Ollama HTTP client replaced by the C-ABI call.  The returned closure
    also carries `.stream(ctx, req, emit)`: the §8f-row-4 streaming form (Done=false frames with text deltas, then
    the Done=true frame) — the reference itself rejects stream:true (api.go:155)."""

    def _request(req: BaseMessage):
        generate_req = req.get_generate_request()
        if generate_req is None:                                     # api.go:48-51
            raise HandlerError("expected GenerateRequest, got different message type")
        return generate_req

    def _raw(generate_req) -> bool:
        # raw = "do not apply the chat template", logprobs = GenerateResponse.logprobs: only the byte-level entry points
        # of libclengine know how
        o = generate_req.options
        return bool(o and (o.raw or o.logprobs) and hasattr(engine, "handle_message_stream"))

    def handler(ctx, req: BaseMessage) -> BaseMessage:
        generate_req = _request(req)
        if _raw(generate_req):
            return worker_api_handler_bytes(engine, sampling)(ctx, req)
        try:
            r = engine.generate(generate_req.model, generate_req.prompt, merge_sampling(sampling, generate_req.options))
        except eng.EngineError as ex:                                # api.go:63-68 wraps the backend error
            raise HandlerError(f"failed to call B200 engine: {ex}") from ex
        return _response(generate_req.model, r.text, True, r.done_reason)

    def stream(ctx, req: BaseMessage, emit) -> None:
        generate_req = _request(req)
        if _raw(generate_req):
            return worker_api_handler_bytes(engine, sampling).stream(ctx, req, emit)
        if not hasattr(engine, "generate_stream"):                   # engines without streaming answer in one frame
            return emit(handler(ctx, req))

        def on_text(delta, ids):
            if delta:
                emit(_response(generate_req.model, delta, False))
            return False

        try:
            r = engine.generate_stream(generate_req.model, generate_req.prompt, merge_sampling(sampling, generate_req.options),
                                       on_text)
        except eng.EngineError as ex:
            raise HandlerError(f"failed to call B200 engine: {ex}") from ex
        emit(_response(generate_req.model, "", True, r.done_reason))

    handler.stream = stream
    return handler


def worker_api_handler_bytes(engine: "eng.Engine", sampling: "eng.Sampling | None" = None):
    """Same handler at the byte level: serialised BaseMessage in, serialised BaseMessage out, entirely
    inside libclengine.so (cl_handle_message) — what a non-Go host would bind."""

    def _wrap(ex):
        if ex.status == eng.CL_ERR_BAD_MESSAGE:
            return HandlerError("expected GenerateRequest, got different message type")
        return HandlerError(f"failed to call B200 engine: {ex}")

    def handler(ctx, req: BaseMessage) -> BaseMessage:
        try:
            return BaseMessage.decode(engine.handle_message(req.encode(), sampling))
        except eng.EngineError as ex:
            raise _wrap(ex) from ex

    def stream(ctx, req: BaseMessage, emit) -> None:
        try:
            engine.handle_message_stream(req.encode(), sampling, lambda frame: emit(BaseMessage.decode(frame)) and False)
        except eng.EngineError as ex:
            raise _wrap(ex) from ex

    handler.stream = stream
    return handler


def default_api_handler(ctx, req: BaseMessage) -> BaseMessage:       # api.go:163-189
    generate_req = req.get_generate_request()
    if generate_req is None:
        raise HandlerError("expected GenerateRequest, got different message type")
    now = time.time_ns()
    return BaseMessage(generate_response=GenerateResponse(
        model=generate_req.model, created_at_seconds=now // 10**9, created_at_nanos=now % 10**9,
        response=f"Generated response for model {generate_req.model} with prompt: {generate_req.prompt}",
        done=True, done_reason="stop", worker_id="default-worker", total_duration=now))


def create_generate_request(model: str, prompt: str, stream: bool, options=None) -> BaseMessage:       # api.go:192-204
    return BaseMessage(generate_request=GenerateRequest(model=model, prompt=prompt, stream=stream, options=options))


def extract_generate_request(msg: BaseMessage) -> GenerateRequest:                       # api.go:207-213
    if msg.get_generate_request() is None:
        raise HandlerError("message does not contain a GenerateRequest")
    return msg.generate_request


def extract_generate_response(msg: BaseMessage) -> GenerateResponse:                     # api.go:216-222
    if msg.get_generate_response() is None:
        raise HandlerError("message does not contain a GenerateResponse")
    return msg.generate_response


def handle_inference_stream(handler: UnifiedAPIHandler, stream, worker_mode: bool = True, ctx=None) -> bool:
    """Peer.handleInferenceRequest (peer.go:190-256): read one length-prefixed request, call the
    handler, turn a handler error into Response="Error: ...", Done=true (peer.go:232-243), write the
    length-prefixed response.  Returns False when the request was dropped (non-worker / unreadable)."""
    if not worker_mode:                                              # peer.go:200-203
        return False
    try:
        req = read_length_prefixed_pb(stream)                        # peer.go:206-210
    except Exception:
        return False
    gr = req.get_generate_request()
    if gr is not None and gr.stream and hasattr(handler, "stream"):
        # streaming extension: several length-prefixed frames on the same stream, the last one has Done=true
        try:
            handler.stream(ctx, req, lambda m: write_length_prefixed_pb(stream, m))
        except Exception as ex:
            write_length_prefixed_pb(stream, BaseMessage(generate_response=GenerateResponse(response=f"Error: {ex}", done=True)))
        return True
    try:
        resp = handler(ctx, req)
    except Exception as ex:                                          # peer.go:232-243
        resp = BaseMessage(generate_response=GenerateResponse(response=f"Error: {ex}", done=True))
    write_length_prefixed_pb(stream, resp)                           # peer.go:248
    return True
