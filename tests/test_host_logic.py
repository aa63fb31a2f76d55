"""CPU-only tests: the C-ABI library loads and exports every declared symbol, the paged-KV allocator,
framing / protobuf codec (mirrors /root/reference/pkg/crowdllama/pbwire_test.go), the handler
envelope with a mock engine (mirrors /root/reference/pkg/ipc/ipc_test.go:44-146), routing
(manager.go:338-387) and Resource JSON (types_test.go)."""
import collections
import io
import json
import os
import random
import re
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import pytest

from crowdllama_b200 import engine as eng
from crowdllama_b200 import handler as H
from crowdllama_b200 import pbwire
from crowdllama_b200.pb import BaseMessage, GenerateRequest, GenerateResponse
from crowdllama_b200.router import Resource, find_best_worker

ROOT = Path(__file__).resolve().parents[1]


# ---- C-ABI ---------------------------------------------------------------------------------------
def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "clengine.h").read_text()
    body = re.sub(r"/\*.*?\*/", "", header, flags=re.S)              # strip comments
    declared = set(re.findall(r"\b(cl_[a-z0-9_]+)\s*\(", body))
    L = eng.lib()
    missing = [s for s in sorted(declared) if not hasattr(L, s)]
    assert not missing, missing
    assert declared == set(eng.EXPORTS), declared ^ set(eng.EXPORTS)
    assert L.cl_abi_version() == 2
    assert b"GenerateRequest" in L.cl_strerror(eng.CL_ERR_BAD_MESSAGE)


def test_presets_and_defaults():
    p = eng.model_preset("llama3-8b")
    assert (p["n_layers"], p["d_model"], p["n_heads"], p["n_kv_heads"], p["head_dim"], p["d_ff"], p["vocab_size"]) == \
        (32, 4096, 32, 8, 128, 14336, 128256)
    assert eng.model_preset("mistral-7b")["vocab_size"] == 32000
    assert eng.model_preset("tinyllama-1.1b")["n_kv_heads"] == 4
    with pytest.raises(eng.EngineError):
        eng.model_preset("nope")
    s = eng.ollama_default_sampling(seed=1)
    assert (round(s.temperature, 3), s.top_k, round(s.top_p, 3), round(s.repeat_penalty, 3), s.repeat_last_n) == (0.8, 40, 0.9, 1.1, 64)
    g = eng.greedy(5)
    assert g.temperature == 0 and g.max_new_tokens == 5


_NO_DEVICE_CHILD = """
import numpy as np
from crowdllama_b200 import engine as eng
assert eng.device_count() == 0
for call in (lambda: eng.Engine(preset="tiny-test"), lambda: eng.op_gemv(np.zeros((2, 16), np.uint16), np.zeros(16, np.float32))):
    try:
        call()
    except eng.EngineError as ex:
        assert ex.status == eng.CL_ERR_NO_DEVICE, ex.status
    else:
        raise AssertionError("the call succeeded without a device")
"""


def test_no_cpu_fallback():
    """Without a device the product path must fail loudly (never route to the oracle).  The device-facing calls run in
    a child process that sees no GPU, so the check holds on machines with and without one."""
    r = subprocess.run([sys.executable, "-c", _NO_DEVICE_CHILD], cwd=ROOT, env={**os.environ, "CUDA_VISIBLE_DEVICES": ""},
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-2000:]
    src = "".join(p.read_text() for p in (ROOT / "crowdllama_b200").rglob("*.py"))
    assert "oracle" not in src.replace("oracle oc_sample", "").replace("the oracle", "")


# ---- paged-KV allocator ------------------------------------------------------------------------------
def test_kvpool_reserve_release_and_oom():
    p = eng.KvPool(8, 16)
    assert p.free_pages == 8
    assert p.reserve(1, 1) == 0 and p.pages_of(1) == [0]
    assert p.reserve(1, 16) == 0 and len(p.pages_of(1)) == 1
    assert p.reserve(1, 17) == 0 and p.pages_of(1) == [0, 1]
    assert p.reserve(2, 16 * 5) == 0 and p.used_pages == 7
    assert p.reserve(3, 33) == eng.CL_ERR_OOM            # needs 3, only 1 free
    assert p.pages_of(3) == [] and p.free_pages == 1     # atomic: nothing taken
    assert p.release(2) == 0 and p.free_pages == 6
    assert p.reserve(3, 33) == 0
    all_pages = p.pages_of(1) + p.pages_of(3)
    assert len(set(all_pages)) == len(all_pages)
    assert p.release(1) == 0 and p.release(3) == 0 and p.free_pages == 8
    assert p.release(99) == 0


def test_kvpool_randomised_never_double_allocates():
    rng = random.Random(0)
    p = eng.KvPool(64, 32)
    want = {}
    for _ in range(2000):
        o = rng.randrange(10)
        if rng.random() < 0.3:
            p.release(o)
            want.pop(o, None)
        else:
            n = rng.randrange(1, 400)
            rc = p.reserve(o, n)
            if rc == 0:
                want[o] = max(want.get(o, 0), (n + 31) // 32)
        owned = [pg for o2 in want for pg in p.pages_of(o2)]
        assert len(owned) == len(set(owned)) == p.used_pages
        for o2, cnt in want.items():
            assert len(p.pages_of(o2)) == cnt


# ---- framing + codec (pbwire_test.go) ----------------------------------------------------------------
def test_length_prefixed_round_trip_request_and_response():
    buf = io.BytesIO()
    req = H.create_generate_request("test-model", "Hello, world!", False)
    pbwire.write_length_prefixed_pb(buf, req)
    raw = buf.getvalue()
    assert int.from_bytes(raw[:4], "big") == len(raw) - 4
    got = pbwire.read_length_prefixed_pb(io.BytesIO(raw))
    r = H.extract_generate_request(got)
    assert (r.model, r.prompt, r.stream) == ("test-model", "Hello, world!", False)
    resp = BaseMessage(generate_response=GenerateResponse(model="test-model", response="Hello back!", done=True,
                                                          done_reason="stop", worker_id="worker", total_duration=123,
                                                          created_at_seconds=1700000000, created_at_nanos=5))
    buf = io.BytesIO()
    pbwire.write_length_prefixed_pb(buf, resp)
    g = H.extract_generate_response(pbwire.read_length_prefixed_pb(io.BytesIO(buf.getvalue())))
    assert g == resp.generate_response
    with pytest.raises(H.HandlerError):
        H.extract_generate_request(resp)


def test_read_rejects_oversize_and_truncated():
    with pytest.raises(ValueError, match="message too large"):
        pbwire.read_length_prefixed_pb(io.BytesIO((10 * 1024 * 1024 + 1).to_bytes(4, "big")))
    with pytest.raises(IOError, match="failed to read length prefix"):
        pbwire.read_length_prefixed_pb(io.BytesIO(b"\x00\x00"))
    with pytest.raises(IOError, match="failed to read protobuf data"):
        pbwire.read_length_prefixed_pb(io.BytesIO((100).to_bytes(4, "big") + b"abc"))


def test_codec_is_wire_compatible_with_google_protobuf():
    """Build llama.v1 descriptors at run time with the protobuf runtime (same field table) and check
    that bytes cross-parse both ways."""
    from google.protobuf import descriptor_pb2, descriptor_pool, message_factory, timestamp_pb2  # noqa: F401
    fd = descriptor_pb2.FileDescriptorProto(name="llama_v1_test.proto", package="llama.v1t", syntax="proto3",
                                            dependency=["google/protobuf/timestamp.proto"])
    T = descriptor_pb2.FieldDescriptorProto
    gr = fd.message_type.add(name="GenerateRequest")
    gr.field.add(name="model", number=1, type=T.TYPE_STRING, label=T.LABEL_OPTIONAL)
    gr.field.add(name="prompt", number=2, type=T.TYPE_STRING, label=T.LABEL_OPTIONAL)
    gr.field.add(name="stream", number=3, type=T.TYPE_BOOL, label=T.LABEL_OPTIONAL)
    gr.field.add(name="options", number=4, type=T.TYPE_MESSAGE, type_name=".llama.v1t.GenerateOptions", label=T.LABEL_OPTIONAL)
    go = fd.message_type.add(name="GenerateOptions")          # the §8f-row-3 extension: proto3 `optional` scalars
    for i, (nm, ty) in enumerate([("seed", T.TYPE_UINT64), ("temperature", T.TYPE_FLOAT), ("top_k", T.TYPE_INT32),
                                  ("top_p", T.TYPE_FLOAT), ("repeat_penalty", T.TYPE_FLOAT), ("repeat_last_n", T.TYPE_INT32),
                                  ("num_predict", T.TYPE_INT32), ("raw", T.TYPE_BOOL)]):
        go.oneof_decl.add(name=f"_{nm}")
        go.field.add(name=nm, number=i + 1, type=ty, label=T.LABEL_OPTIONAL, oneof_index=i, proto3_optional=True)
    gp = fd.message_type.add(name="GenerateResponse")
    gp.field.add(name="model", number=1, type=T.TYPE_STRING, label=T.LABEL_OPTIONAL)
    gp.field.add(name="created_at", number=2, type=T.TYPE_MESSAGE, type_name=".google.protobuf.Timestamp", label=T.LABEL_OPTIONAL)
    gp.field.add(name="response", number=3, type=T.TYPE_STRING, label=T.LABEL_OPTIONAL)
    gp.field.add(name="done", number=4, type=T.TYPE_BOOL, label=T.LABEL_OPTIONAL)
    gp.field.add(name="done_reason", number=5, type=T.TYPE_STRING, label=T.LABEL_OPTIONAL)
    gp.field.add(name="worker_id", number=6, type=T.TYPE_STRING, label=T.LABEL_OPTIONAL)
    gp.field.add(name="total_duration", number=7, type=T.TYPE_INT64, label=T.LABEL_OPTIONAL)
    bm = fd.message_type.add(name="BaseMessage")
    bm.oneof_decl.add(name="message")
    bm.field.add(name="generate_request", number=1, type=T.TYPE_MESSAGE, type_name=".llama.v1t.GenerateRequest",
                 label=T.LABEL_OPTIONAL, oneof_index=0)
    bm.field.add(name="generate_response", number=2, type=T.TYPE_MESSAGE, type_name=".llama.v1t.GenerateResponse",
                 label=T.LABEL_OPTIONAL, oneof_index=0)
    pool = descriptor_pool.Default()
    try:
        pool.Add(fd)
    except TypeError:
        pass
    Base = message_factory.GetMessageClass(pool.FindMessageTypeByName("llama.v1t.BaseMessage"))
    ours = H.create_generate_request("tinyllama", "why is the sky blue? ☃", True).encode()
    g = Base.FromString(ours)
    assert g.WhichOneof("message") == "generate_request"
    assert (g.generate_request.model, g.generate_request.prompt, g.generate_request.stream) == ("tinyllama", "why is the sky blue? ☃", True)
    # request options: explicit presence both ways (temperature 0.0 and num_predict -1 must survive)
    from crowdllama_b200.pb import GenerateOptions
    opts = GenerateOptions(seed=(1 << 63) + 5, temperature=0.0, top_k=40, top_p=0.5, num_predict=-1, raw=True)
    g = Base.FromString(H.create_generate_request("m", "p", True, opts).encode())
    o = g.generate_request.options
    assert o.HasField("temperature") and o.temperature == 0.0 and o.seed == (1 << 63) + 5 and o.top_k == 40
    assert o.num_predict == -1 and o.raw and abs(o.top_p - 0.5) < 1e-7
    assert not o.HasField("repeat_penalty") and not o.HasField("repeat_last_n")
    g3 = Base()
    g3.generate_request.model = "m"
    g3.generate_request.options.temperature = 0.0
    g3.generate_request.options.repeat_last_n = 64
    g3.generate_request.options.num_predict = -2
    back_o = BaseMessage.decode(g3.SerializeToString()).generate_request.options
    assert back_o == GenerateOptions(temperature=0.0, repeat_last_n=64, num_predict=-2)
    assert BaseMessage.decode(H.create_generate_request("m", "p", False).encode()).generate_request.options is None
    g2 = Base()
    g2.generate_response.model = "m"
    g2.generate_response.response = "text"
    g2.generate_response.done = True
    g2.generate_response.done_reason = "length"
    g2.generate_response.worker_id = "worker"
    g2.generate_response.total_duration = 1 << 60
    g2.generate_response.created_at.seconds = 1700000001
    g2.generate_response.created_at.nanos = 999
    back = BaseMessage.decode(g2.SerializeToString()).generate_response
    assert back == GenerateResponse("m", 1700000001, 999, "text", True, "length", "worker", 1 << 60)
    assert Base.FromString(BaseMessage(generate_response=back).encode()) == g2


# ---- handler envelope with a mock engine (ipc_test.go:44-146) -----------------------------------------
class _MockEngine:
    model_name = "test-model"

    def generate(self, model, prompt, sampling=None):
        class R:
            text, done_reason = "PB Hello, " + prompt, "stop"
        if model != self.model_name:
            raise eng.EngineError.__new__(eng.EngineError)
        return R()


def test_worker_handler_envelope():
    h = H.worker_api_handler(_MockEngine())
    resp = h(None, H.create_generate_request("test-model", "world", False))
    g = H.extract_generate_response(resp)
    assert g.model == "test-model" and g.response == "PB Hello, world" and g.done and g.done_reason == "stop"
    assert g.worker_id == "worker" and g.total_duration > 0 and g.created_at_seconds > 0
    with pytest.raises(H.HandlerError, match="expected GenerateRequest, got different message type"):
        h(None, BaseMessage(generate_response=GenerateResponse()))


def test_request_options_override_worker_defaults_field_by_field():
    from crowdllama_b200.pb import GenerateOptions
    seen = {}

    class Rec(_MockEngine):
        def generate(self, model, prompt, sampling=None):
            seen["s"] = sampling
            return super().generate(model, prompt, sampling)

    base = eng.Sampling()
    base.temperature, base.top_k, base.top_p, base.repeat_penalty, base.repeat_last_n, base.seed, base.max_new_tokens = 0.8, 40, 0.9, 1.1, 64, 11, 128
    h = H.worker_api_handler(Rec(), base)
    h(None, H.create_generate_request("test-model", "x", False))
    assert seen["s"] is base                                           # no options: the worker's defaults, untouched
    h(None, H.create_generate_request("test-model", "x", False, GenerateOptions(temperature=0.0, seed=5, num_predict=7)))
    s = seen["s"]
    assert (s.temperature, s.seed, s.max_new_tokens) == (0.0, 5, 7)
    assert (s.top_k, s.repeat_last_n) == (40, 64) and abs(s.top_p - 0.9) < 1e-6 and abs(s.repeat_penalty - 1.1) < 1e-6
    assert base.temperature == pytest.approx(0.8) and base.seed == 11  # the default object is not mutated


def test_raw_requests_take_the_byte_level_entry_point():
    """options.raw (no chat template) is implemented inside libclengine: the closure hands such requests over as bytes."""
    from crowdllama_b200.pb import GenerateOptions
    seen = []

    class Bytes(_MockEngine):
        def handle_message(self, req, sampling=None):
            seen.append(BaseMessage.decode(req).generate_request)
            return H._response("test-model", "raw answer", True, "stop").encode()

        def handle_message_stream(self, req, sampling=None, on_frame=None):
            on_frame(H._response("test-model", "raw ", False).encode())
            on_frame(H._response("test-model", "", True, "length").encode())
            return 2

    h = H.worker_api_handler(Bytes())
    g = h(None, H.create_generate_request("test-model", "p", False, GenerateOptions(raw=True, temperature=0.0))).generate_response
    assert g.response == "raw answer" and seen[0].options.raw and seen[0].options.temperature == 0.0
    assert h(None, H.create_generate_request("test-model", "p", False, GenerateOptions(temperature=0.0))).generate_response.response == "PB Hello, p"
    frames = []
    h.stream(None, H.create_generate_request("test-model", "p", True, GenerateOptions(raw=True)), frames.append)
    assert [f.generate_response.done for f in frames] == [False, True] and frames[-1].generate_response.done_reason == "length"


def test_streaming_frames_on_the_inference_stream():
    """SURVEY.md §8f row 4: stream=true -> several length-prefixed GenerateResponse frames, Done only on the last."""
    class Duplex(io.BytesIO):
        def __init__(self, data):
            super().__init__(data)
            self.out = io.BytesIO()

        def write(self, b):
            return self.out.write(b)

    class Streaming(_MockEngine):
        def generate_stream(self, model, prompt, sampling=None, on_text=None):
            for piece in ("PB ", "Hello, ", "", prompt):
                on_text(piece, [1])
            return self.generate(model, prompt, sampling)

    def frames(handler, stream_flag):
        wire = io.BytesIO()
        pbwire.write_length_prefixed_pb(wire, H.create_generate_request("test-model", "world", stream_flag))
        s = Duplex(wire.getvalue())
        assert H.handle_inference_stream(handler, s)
        rd, out = io.BytesIO(s.out.getvalue()), []
        while rd.tell() < len(rd.getvalue()):
            out.append(pbwire.read_length_prefixed_pb(rd).generate_response)
        return out

    fs = frames(H.worker_api_handler(Streaming()), True)
    assert [f.response for f in fs] == ["PB ", "Hello, ", "world", ""]  # empty deltas are not sent; the last frame closes
    assert [f.done for f in fs] == [False, False, False, True] and fs[-1].done_reason == "stop"
    assert all(f.model == "test-model" and f.worker_id == "worker" for f in fs) and fs[0].total_duration == 0
    assert len(frames(H.worker_api_handler(Streaming()), False)) == 1   # stream=false: the reference's single answer
    one = frames(H.worker_api_handler(_MockEngine()), True)             # an engine without streaming: one complete frame
    assert len(one) == 1 and one[0].done and one[0].response == "PB Hello, world"

    def failing_stream(ctx, req, emit):
        emit(H._response("test-model", "partial", False))
        raise RuntimeError("boom")
    h = H.worker_api_handler(Streaming())
    h.stream = failing_stream
    fs = frames(h, True)
    assert fs[-1].response == "Error: boom" and fs[-1].done            # peer.go:232-243 semantics, mid-stream


def test_handle_inference_stream_error_becomes_text():
    class Duplex(io.BytesIO):
        def __init__(self, data):
            super().__init__(data)
            self.out = io.BytesIO()

        def write(self, b):
            return self.out.write(b)

    def failing(ctx, req):
        raise RuntimeError("boom")
    wire = io.BytesIO()
    pbwire.write_length_prefixed_pb(wire, H.create_generate_request("m", "p", False))
    s = Duplex(wire.getvalue())
    assert H.handle_inference_stream(failing, s)
    g = pbwire.read_length_prefixed_pb(io.BytesIO(s.out.getvalue())).generate_response
    assert g.response == "Error: boom" and g.done and g.model == ""        # peer.go:235-242
    assert not H.handle_inference_stream(failing, Duplex(b""), worker_mode=False)
    assert not H.handle_inference_stream(failing, Duplex(b"\x00"))
    s = Duplex(wire.getvalue())
    assert H.handle_inference_stream(H.default_api_handler, s)
    g = pbwire.read_length_prefixed_pb(io.BytesIO(s.out.getvalue())).generate_response
    assert g.response == "Generated response for model m with prompt: p" and g.worker_id == "default-worker"


# ---- routing (manager.go:338-387) and Resource JSON (types_test.go) -----------------------------------
def _w(pid, models, tput, load, worker=True):
    return Resource(peer_id=pid, supported_models=models, tokens_throughput=tput, load=load, worker_mode=worker)


def test_find_best_worker_rule():
    ws = [_w("a", ["tinyllama"], 150, 0.3), _w("b", ["tinyllama", "llama3:8b"], 300, 0.5), _w("c", ["llama3:8b"], 100, 0.0),
          _w("consumer", ["llama3:8b"], 1e9, 0.0, worker=False)]
    assert find_best_worker(ws, "llama3:8b").peer_id == "b"        # 200 > 100
    assert find_best_worker(ws, "tinyllama").peer_id == "b"        # 200 > 115.4
    assert find_best_worker(ws, "llama3") is None                  # exact string match only
    assert find_best_worker([], "x") is None
    assert find_best_worker([_w("z", ["m"], 0.0, 0.0)], "m") is None   # score 0 never beats bestScore 0 (strict >)


def test_ties_are_uniform_random():
    ws = [_w(str(i), ["m"], 150.0, 0.3) for i in range(8)]
    rng = random.Random(0)
    counts = {}
    for _ in range(4000):
        p = find_best_worker(ws, "m", rng).peer_id
        counts[p] = counts.get(p, 0) + 1
    assert len(counts) == 8 and min(counts.values()) > 350


def test_advertised_throughput_buckets_make_identical_workers_tie():
    from crowdllama_b200.router import advertised_throughput
    assert advertised_throughput(0.0) == 0.0
    a, b = advertised_throughput(3190.0), advertised_throughput(3260.0)       # two B200s, EWMAs 2 % apart
    assert a == b and 2700 < a < 3900
    assert advertised_throughput(5700.0) > a                                  # an idle worker (short steps) still ranks higher
    ws = [_w(f"w{i}", ["m"], advertised_throughput(3200.0 + 13 * i), 0.0) for i in range(4)]
    picks = collections.Counter(find_best_worker(ws, "m", random.Random(s)).peer_id for s in range(400))
    assert len(picks) == 4 and min(picks.values()) > 60                       # ties -> uniform random, as with the constant 150


def test_resource_json_round_trip():
    r = _w("12D3KooW", ["llama3:8b"], 301.5, 0.25)
    r.vram_gb, r.gpu_model = 179, "NVIDIA B200"
    d = json.loads(r.to_json())
    assert set(d) == {"peer_id", "supported_models", "tokens_throughput", "vram_gb", "load", "gpu_model", "last_updated",
                      "version", "worker_mode"}
    assert Resource.from_json(r.to_json()) == r
    assert r.get_dht_key() == "/ipns/12D3KooW"
    with pytest.raises(ValueError, match="failed to unmarshal CrowdLlamaResource"):
        Resource.from_json(b"{nope")


def test_checkpoint_validation_is_host_logic(tmp_path):
    """csrc/weights_io.cpp without a GPU: config.json + safetensors headers of the HF-written fixture
    (tests/golden/hf_tiny_llama_ckpt) and of hand-written F32 / sharded / broken variants."""
    import numpy as np
    from st_util import hf_tensors_from_fixture, write_safetensors
    G = Path(__file__).resolve().parent / "golden"
    cfg, nt, npar = eng.checkpoint_info(G / "hf_tiny_llama_ckpt")
    assert (cfg["n_layers"], cfg["d_model"], cfg["n_heads"], cfg["n_kv_heads"], cfg["head_dim"], cfg["d_ff"], cfg["vocab_size"]) == \
           (2, 128, 2, 1, 64, 256, 256)
    assert abs(cfg["rope_theta"] - 1e4) < 1e-3 and nt == 3 + 2 * 9
    z = np.load(G / "hf_tiny_llama.npz")
    tensors = hf_tensors_from_fixture(z, cfg)
    assert npar == sum(int(np.prod(shape)) for _, shape in tensors.values())
    write_safetensors(tmp_path / "f32.safetensors", tensors, "F32")
    assert eng.checkpoint_info(tmp_path / "f32.safetensors", cfg)[1:] == (nt, npar)
    # tied embeddings: lm_head is synthesised from embed_tokens
    tied = {k: v for k, v in tensors.items() if k != "lm_head.weight"}
    write_safetensors(tmp_path / "tied.safetensors", tied)
    assert eng.checkpoint_info(tmp_path / "tied.safetensors", cfg)[1] == nt
    # broken inputs fail with CL_ERR_IO and a message naming the tensor
    missing = {k: v for k, v in tensors.items() if k != "model.layers.1.mlp.up_proj.weight"}
    write_safetensors(tmp_path / "missing.safetensors", missing)
    with pytest.raises(eng.EngineError) as ei:
        eng.checkpoint_info(tmp_path / "missing.safetensors", cfg)
    assert ei.value.status == eng.CL_ERR_IO and "L1:10" in ei.value.detail
    wrong = dict(cfg); wrong["n_kv_heads"] = 2
    with pytest.raises(eng.EngineError) as ei:
        eng.checkpoint_info(tmp_path / "f32.safetensors", wrong)
    assert "k_proj" in ei.value.detail
    raw = (tmp_path / "f32.safetensors").read_bytes()
    (tmp_path / "trunc.safetensors").write_bytes(raw[: len(raw) // 2])
    with pytest.raises(eng.EngineError):
        eng.checkpoint_info(tmp_path / "trunc.safetensors", cfg)
    (tmp_path / "garbage.safetensors").write_bytes(b"\xff" * 64)
    with pytest.raises(eng.EngineError):
        eng.checkpoint_info(tmp_path / "garbage.safetensors", cfg)
    with pytest.raises(eng.EngineError):
        eng.checkpoint_info(tmp_path, None)                     # a directory without config.json


def test_advertised_metadata_rule():
    """INTEGRATION.md "What to advertise": capacity in half-octave buckets (identical workers tie), Load flagged only
    once a whole extra batch waits."""
    from crowdllama_b200 import router
    assert router.advertised_throughput(11000.0) == router.advertised_throughput(12500.0)
    assert router.advertised_throughput(11000.0) != router.advertised_throughput(22000.0)
    assert router.advertised_throughput(0.0) == 0.0
    assert [router.advertised_load(x) for x in (0.0, 0.99, 1.0, 1.9, 2.0, 7.5)] == [0.0, 0.0, 0.0, 0.0, 1.0, 1.0]


def _hf_filtered_probs(logits, history, temperature, top_k, top_p, penalty):
    """The same chain built from the HF transformers logits processors (an independent implementation of every stage):
    repetition penalty -> top-k -> temperature -> top-p, then softmax over what is left."""
    import torch
    from transformers.generation.logits_process import (RepetitionPenaltyLogitsProcessor, TemperatureLogitsWarper, TopKLogitsWarper,
                                                         TopPLogitsWarper)
    sc = torch.tensor(np.asarray(logits, np.float32))[None, :].double()
    ids = torch.tensor(list(history), dtype=torch.long)[None, :] if len(history) else torch.zeros((1, 0), dtype=torch.long)
    if penalty != 1.0 and len(history):
        sc = RepetitionPenaltyLogitsProcessor(penalty)(ids, sc)
    if top_k > 0:
        sc = TopKLogitsWarper(top_k)(ids, sc)
    sc = TemperatureLogitsWarper(temperature)(ids, sc)
    if 0.0 < top_p < 1.0:
        sc = TopPLogitsWarper(top_p)(ids, sc)
    return torch.softmax(sc, dim=-1)[0].numpy()


@pytest.mark.parametrize("case", [
    dict(temperature=0.8, top_k=40, top_p=0.9, penalty=1.1, hist=24),     # Ollama's defaults (api.go:109-118 sends no options)
    dict(temperature=1.3, top_k=0, top_p=0.7, penalty=1.0, hist=0),       # nucleus only
    dict(temperature=0.5, top_k=5, top_p=1.0, penalty=1.6, hist=10),      # top-k only, strong penalty
    dict(temperature=1.0, top_k=12, top_p=0.5, penalty=1.3, hist=40),
])
def test_sampler_stages_match_hf_logits_processors(case):
    """Pins the sampler (the library's cl_sample_token AND the CPU checker's) to an implementation that is not this
    repository's: support set and probabilities of the HF transformers processors applied in the same order.  8000
    draws per case over a 64-token vocabulary: no draw outside HF's support, every token's frequency within 5 sigma."""
    from oracle import oracle as oc
    rng = np.random.default_rng(zlib.crc32(repr(sorted(case.items())).encode()))   # hash() of a str varies per process
    V, n = 64, 8000
    lg = (rng.standard_normal(V) * 2.0).astype(np.float32)
    hist = [int(x) for x in rng.integers(0, V, size=case["hist"])]
    p = _hf_filtered_probs(lg, hist, case["temperature"], case["top_k"], case["top_p"], case["penalty"])
    sp = eng.ollama_default_sampling(seed=4242)
    sp.temperature, sp.top_k, sp.top_p, sp.repeat_penalty, sp.repeat_last_n = case["temperature"], case["top_k"], case["top_p"], case["penalty"], 64
    ours = np.bincount([eng.sample_token(lg, sp, hist, step=i) for i in range(n)], minlength=V)
    chk = np.bincount([oc.sample(lg, case["temperature"], case["top_k"], case["top_p"], case["penalty"], 64, seed=4242, history=hist, step=i)
                       for i in range(n)], minlength=V)
    assert (ours == chk).all()                                   # library sampler == CPU checker, draw by draw
    assert ours[p == 0].sum() == 0, "a token outside the HF support set was drawn"
    sigma = np.sqrt(n * p * (1 - p)) + 1e-9
    assert (np.abs(ours - n * p) <= 5 * sigma + 1).all(), (ours, n * p)
    assert (p > 0).sum() >= 2                                    # the case exercises a real distribution


def test_checkpoint_config_rejects_what_the_engine_does_not_implement(tmp_path):
    """config.json features that would change the tokens must fail loudly (scaled RoPE, another activation, biases); a
    sliding attention window is honoured by capping the served context at the window."""
    import json
    import shutil
    import numpy as np
    from st_util import write_safetensors
    G = Path(__file__).resolve().parent / "golden" / "hf_tiny_llama_ckpt"
    base = json.loads((G / "config.json").read_text())

    def variant(name, **changes):
        d = tmp_path / name
        d.mkdir()
        shutil.copy(G / "model.safetensors", d / "model.safetensors")
        cfg = dict(base)
        cfg.update(changes)
        (d / "config.json").write_text(json.dumps(cfg))
        return d
    assert eng.checkpoint_info(variant("plain"))[0]["max_seq_len"] == 64
    assert eng.checkpoint_info(variant("swa", sliding_window=32))[0]["max_seq_len"] == 32          # Mistral-7B-v0.1 style
    assert eng.checkpoint_info(variant("swa_none", sliding_window=None))[0]["max_seq_len"] == 64
    assert eng.checkpoint_info(variant("old_style", rope_parameters=None, rope_theta=500000.0, rope_scaling=None))[0]["rope_theta"] == 500000.0
    c31 = eng.checkpoint_info(variant("llama31", rope_parameters={"rope_theta": 500000.0, "rope_type": "llama3", "factor": 8.0, "low_freq_factor": 1.0,
                                                                   "high_freq_factor": 4.0, "original_max_position_embeddings": 8192}))[0]
    assert (c31["rope_factor"], c31["rope_low_freq_factor"], c31["rope_high_freq_factor"], c31["rope_original_max_pos"]) == (8.0, 1.0, 4.0, 8192)
    for name, changes, needle in [
            ("yarn", dict(rope_parameters={"rope_theta": 500000.0, "rope_type": "yarn", "factor": 8.0}), "yarn"),
            ("llama3_incomplete", dict(rope_parameters={"rope_theta": 500000.0, "rope_type": "llama3", "factor": 8.0}), "llama3 needs"),
            ("linear", dict(rope_parameters=None, rope_theta=10000.0, rope_scaling={"type": "linear", "factor": 2.0}), "linear"),
            ("gelu", dict(hidden_act="gelu"), "hidden_act"),
            ("bias", dict(attention_bias=True), "attention_bias")]:
        with pytest.raises(eng.EngineError) as ei:
            eng.checkpoint_info(variant(name, **changes))
        assert ei.value.status == eng.CL_ERR_IO and needle in ei.value.detail, ei.value.detail
    # a bias tensor in the file itself (Qwen-style checkpoints) is refused, not ignored
    cfg, _, _ = eng.checkpoint_info(G)
    from st_util import hf_tensors_from_fixture
    t = hf_tensors_from_fixture(np.load(G.parent / "hf_tiny_llama.npz"), cfg)
    t["model.layers.0.self_attn.q_proj.bias"] = (np.zeros(128, np.uint16), (128,))
    write_safetensors(tmp_path / "with_bias.safetensors", t)
    with pytest.raises(eng.EngineError) as ei:
        eng.checkpoint_info(tmp_path / "with_bias.safetensors", cfg)
    assert "q_proj.bias" in ei.value.detail


def test_graft_entry_build_check():
    """The driver's "does it build" hook: compiles (incrementally) and checks the ABI version the binding expects."""
    import importlib
    g = importlib.import_module("__graft_entry__")
    g.build()
