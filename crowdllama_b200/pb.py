"""Minimal protobuf codec for llama.v1.BaseMessage — the wire schema of the reference's inference
protocol (external module github.com/crowdllama/crowdllama-pb, /root/reference/go.mod:6).

That module is not vendored, so field NUMBERS are an assumption kept in ONE table here (and
mirrored in csrc/host_util.cpp): the declaration order of the Go struct literals at
/root/reference/pkg/crowdllama/api.go:77-85 and :193-197.  Field NAMES are the reference's.
"""
from __future__ import annotations

from dataclasses import dataclass, field

FIELDS = {
    "BaseMessage": {"generate_request": 1, "generate_response": 2},
    "GenerateRequest": {"model": 1, "prompt": 2, "stream": 3, "options": 4},
    # EXTENSION (SURVEY.md §8f row 3): request options the reference's wire cannot express (api.go:193-197);
    # every field has explicit presence (proto3 `optional`): temperature 0 = greedy is not "unset"
    # logprobs / top_logprobs: the log-probabilities of the generated tokens (Ollama's top-level request fields)
    "GenerateOptions": {"seed": 1, "temperature": 2, "top_k": 3, "top_p": 4, "repeat_penalty": 5, "repeat_last_n": 6,
                        "num_predict": 7, "raw": 8, "logprobs": 9, "top_logprobs": 10},
    # EXTENSION: logprobs = one TokenLogprob per token id the frame covers (a peer without it skips field 8)
    "GenerateResponse": {"model": 1, "created_at": 2, "response": 3, "done": 4, "done_reason": 5, "worker_id": 6,
                         "total_duration": 7, "logprobs": 8},
    "TokenLogprob": {"token": 1, "logprob": 2, "top_logprobs": 3},
    "TopLogprob": {"token": 1, "logprob": 2},
    "Timestamp": {"seconds": 1, "nanos": 2},
}


def _varint(v: int) -> bytes:
    v &= (1 << 64) - 1
    out = bytearray()
    while v >= 0x80:
        out.append((v & 0x7F) | 0x80)
        v >>= 7
    out.append(v)
    return bytes(out)


def _rd_varint(b: bytes, i: int):
    r, shift = 0, 0
    while True:
        if i >= len(b) or shift > 63:
            raise ValueError("truncated varint")
        c = b[i]
        i += 1
        r |= (c & 0x7F) << shift
        if not c & 0x80:
            return r, i
        shift += 7


def _ld(fieldno: int, payload: bytes) -> bytes:
    return _varint(fieldno << 3 | 2) + _varint(len(payload)) + payload


def _fields(b: bytes):
    i = 0
    while i < len(b):
        key, i = _rd_varint(b, i)
        f, wt = key >> 3, key & 7
        if wt == 0:
            v, i = _rd_varint(b, i)
        elif wt == 2:
            n, i = _rd_varint(b, i)
            if i + n > len(b):
                raise ValueError("truncated field")
            v, i = b[i:i + n], i + n
        elif wt == 1:
            if i + 8 > len(b):
                raise ValueError("truncated fixed64 field")
            v, i = b[i:i + 8], i + 8
        elif wt == 5:
            if i + 4 > len(b):
                raise ValueError("truncated fixed32 field")
            v, i = b[i:i + 4], i + 4
        else:
            raise ValueError(f"unsupported wire type {wt}")
        yield f, wt, v


import struct

_OPT_FLOAT = ("temperature", "top_p", "repeat_penalty")
_OPT_BOOL = ("raw", "logprobs")


@dataclass
class GenerateOptions:
    """Ollama `options` subset (api/types.go Options upstream): None = not set (the worker's default applies)."""
    seed: int | None = None
    temperature: float | None = None
    top_k: int | None = None
    top_p: float | None = None
    repeat_penalty: float | None = None
    repeat_last_n: int | None = None
    num_predict: int | None = None
    raw: bool | None = None
    logprobs: bool | None = None
    top_logprobs: int | None = None

    def encode(self) -> bytes:
        F, out = FIELDS["GenerateOptions"], b""
        for name, fno in F.items():
            v = getattr(self, name)
            if v is None:
                continue
            if name in _OPT_FLOAT:
                out += _varint(fno << 3 | 5) + struct.pack("<f", float(v))
            else:
                out += _varint(fno << 3) + _varint(int(v))
        return out

    @classmethod
    def decode(cls, b: bytes) -> "GenerateOptions":
        F, m = FIELDS["GenerateOptions"], cls()
        by_no = {v: k for k, v in F.items()}
        for f, wt, v in _fields(b):
            name = by_no.get(f)
            if name is None:
                continue
            if name in _OPT_FLOAT and wt == 5:
                setattr(m, name, struct.unpack("<f", v)[0])
            elif name not in _OPT_FLOAT and wt == 0:
                if name in _OPT_BOOL:
                    setattr(m, name, bool(v))
                elif name == "seed":
                    m.seed = v
                else:
                    setattr(m, name, v if v < 1 << 63 else v - (1 << 64))
        return m

    @classmethod
    def from_json(cls, d: dict | None) -> "GenerateOptions | None":
        """Ollama request JSON `options` object -> GenerateOptions (unknown keys are ignored, as Ollama does)."""
        if not d:
            return None
        m = cls()
        for k in ("seed", "top_k", "repeat_last_n", "num_predict"):
            if d.get(k) is not None:
                setattr(m, k, int(d[k]))
        for k in _OPT_FLOAT:
            if d.get(k) is not None:
                setattr(m, k, float(d[k]))
        return m

    def is_empty(self) -> bool:
        return all(getattr(self, k) is None for k in FIELDS["GenerateOptions"])


def _f32(fno: int, v: float) -> bytes:
    return _varint(fno << 3 | 5) + struct.pack("<f", float(v)) if v != 0.0 else b""


@dataclass
class TopLogprob:
    token: bytes = b""              # the surface bytes of the id on its own
    logprob: float = 0.0

    def encode(self) -> bytes:
        F = FIELDS["TopLogprob"]
        return (_ld(F["token"], self.token) if self.token else b"") + _f32(F["logprob"], self.logprob)

    @classmethod
    def decode(cls, b: bytes) -> "TopLogprob":
        F, m = FIELDS["TopLogprob"], cls()
        for f, wt, v in _fields(b):
            if f == F["token"] and wt == 2:
                m.token = bytes(v)
            elif f == F["logprob"] and wt == 5:
                m.logprob = struct.unpack("<f", v)[0]
        return m


@dataclass
class TokenLogprob:
    token: bytes = b""
    logprob: float = 0.0
    top_logprobs: list = field(default_factory=list)    # [TopLogprob]

    def encode(self) -> bytes:
        F = FIELDS["TokenLogprob"]
        out = (_ld(F["token"], self.token) if self.token else b"") + _f32(F["logprob"], self.logprob)
        for t in self.top_logprobs:
            out += _ld(F["top_logprobs"], t.encode())
        return out

    @classmethod
    def decode(cls, b: bytes) -> "TokenLogprob":
        F, m = FIELDS["TokenLogprob"], cls()
        for f, wt, v in _fields(b):
            if f == F["token"] and wt == 2:
                m.token = bytes(v)
            elif f == F["logprob"] and wt == 5:
                m.logprob = struct.unpack("<f", v)[0]
            elif f == F["top_logprobs"] and wt == 2:
                m.top_logprobs.append(TopLogprob.decode(v))
        return m


@dataclass
class GenerateRequest:
    model: str = ""
    prompt: str = ""
    stream: bool = False
    options: GenerateOptions | None = None

    def encode(self) -> bytes:
        F = FIELDS["GenerateRequest"]
        out = b""
        if self.model:
            out += _ld(F["model"], self.model.encode())
        if self.prompt:
            out += _ld(F["prompt"], self.prompt.encode())
        if self.stream:
            out += _varint(F["stream"] << 3) + b"\x01"
        if self.options is not None and not self.options.is_empty():
            out += _ld(F["options"], self.options.encode())
        return out

    @classmethod
    def decode(cls, b: bytes) -> "GenerateRequest":
        F, m = FIELDS["GenerateRequest"], cls()
        for f, wt, v in _fields(b):
            if f == F["model"] and wt == 2:
                m.model = v.decode("utf-8", "replace")
            elif f == F["prompt"] and wt == 2:
                m.prompt = v.decode("utf-8", "replace")
            elif f == F["stream"] and wt == 0:
                m.stream = bool(v)
            elif f == F["options"] and wt == 2:
                m.options = GenerateOptions.decode(v)
        return m


@dataclass
class GenerateResponse:
    model: str = ""
    created_at_seconds: int = 0
    created_at_nanos: int = 0
    response: str = ""
    done: bool = False
    done_reason: str = ""
    worker_id: str = ""
    total_duration: int = 0
    logprobs: list = field(default_factory=list)        # [TokenLogprob], one per token id of this frame

    def encode(self) -> bytes:
        F, T = FIELDS["GenerateResponse"], FIELDS["Timestamp"]
        out = b""
        if self.model:
            out += _ld(F["model"], self.model.encode())
        ts = b""
        if self.created_at_seconds:
            ts += _varint(T["seconds"] << 3) + _varint(self.created_at_seconds)
        if self.created_at_nanos:
            ts += _varint(T["nanos"] << 3) + _varint(self.created_at_nanos)
        if ts:
            out += _ld(F["created_at"], ts)
        if self.response:
            out += _ld(F["response"], self.response.encode())
        if self.done:
            out += _varint(F["done"] << 3) + b"\x01"
        if self.done_reason:
            out += _ld(F["done_reason"], self.done_reason.encode())
        if self.worker_id:
            out += _ld(F["worker_id"], self.worker_id.encode())
        if self.total_duration:
            out += _varint(F["total_duration"] << 3) + _varint(self.total_duration)
        for t in self.logprobs:
            out += _ld(F["logprobs"], t.encode())
        return out

    @classmethod
    def decode(cls, b: bytes) -> "GenerateResponse":
        F, T, m = FIELDS["GenerateResponse"], FIELDS["Timestamp"], cls()
        for f, wt, v in _fields(b):
            if f == F["model"] and wt == 2:
                m.model = v.decode("utf-8", "replace")
            elif f == F["created_at"] and wt == 2:
                for f2, wt2, v2 in _fields(v):
                    if f2 == T["seconds"]:
                        m.created_at_seconds = v2
                    elif f2 == T["nanos"]:
                        m.created_at_nanos = v2
            elif f == F["response"] and wt == 2:
                m.response = v.decode("utf-8", "replace")
            elif f == F["done"] and wt == 0:
                m.done = bool(v)
            elif f == F["done_reason"] and wt == 2:
                m.done_reason = v.decode("utf-8", "replace")
            elif f == F["worker_id"] and wt == 2:
                m.worker_id = v.decode("utf-8", "replace")
            elif f == F["total_duration"] and wt == 0:
                m.total_duration = v if v < 1 << 63 else v - (1 << 64)
            elif f == F["logprobs"] and wt == 2:
                m.logprobs.append(TokenLogprob.decode(v))
        return m


@dataclass
class BaseMessage:
    """oneof message { GenerateRequest generate_request; GenerateResponse generate_response; }"""
    generate_request: GenerateRequest | None = None
    generate_response: GenerateResponse | None = None
    unknown: list = field(default_factory=list)

    def encode(self) -> bytes:
        F = FIELDS["BaseMessage"]
        if self.generate_request is not None:
            return _ld(F["generate_request"], self.generate_request.encode())
        if self.generate_response is not None:
            return _ld(F["generate_response"], self.generate_response.encode())
        return b""

    @classmethod
    def decode(cls, b: bytes) -> "BaseMessage":
        F, m = FIELDS["BaseMessage"], cls()
        for f, wt, v in _fields(b):
            if f == F["generate_request"] and wt == 2:
                m.generate_request, m.generate_response = GenerateRequest.decode(v), None
            elif f == F["generate_response"] and wt == 2:
                m.generate_response, m.generate_request = GenerateResponse.decode(v), None
            else:
                m.unknown.append(f)
        return m

    # Go-style getters (nil-safe in the reference: req.GetGenerateRequest())
    def get_generate_request(self):
        return self.generate_request

    def get_generate_response(self):
        return self.generate_response
