"""ctypes binding of libclengine.so — the same C-ABI a Go cgo shim binds (include/clengine.h).

There is no CPU fallback anywhere in this package: if the shared library is missing the import
of the binding fails loudly, and if no sm_100 device is visible `Engine(...)` raises
`EngineError(CL_ERR_NO_DEVICE)`.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libclengine.so"

CL_OK = 0
CL_ERR_INVALID_ARG, CL_ERR_NO_DEVICE, CL_ERR_CUDA, CL_ERR_OOM, CL_ERR_UNKNOWN_MODEL, CL_ERR_TOO_LONG, \
    CL_ERR_BAD_SEQ, CL_ERR_SHUTDOWN, CL_ERR_IO, CL_ERR_INTERNAL, CL_ERR_BAD_MESSAGE = range(-1, -12, -1)

# device sampler limits (include/clengine.h CL_SAMPLE_MAX_TOP_K / CL_SAMPLE_MAX_WINDOW)
SAMPLE_MAX_TOP_K = 128
SAMPLE_MAX_WINDOW = 64
# most alternatives a log-probability entry carries (include/clengine.h CL_MAX_TOP_LOGPROBS)
MAX_TOP_LOGPROBS = 20

KINDS = dict(EMBED=0, LM_HEAD=1, FINAL_NORM=2, ATTN_NORM=3, WQ=4, WK=5, WV=6, WO=7, FFN_NORM=8, WGATE=9, WUP=10,
             WDOWN=11)


class ModelConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("n_layers", "d_model", "n_heads", "n_kv_heads", "head_dim", "d_ff",
                                         "vocab_size", "max_seq_len")] + \
               [("rope_theta", C.c_float), ("rms_eps", C.c_float), ("rope_factor", C.c_float), ("rope_low_freq_factor", C.c_float),
                ("rope_high_freq_factor", C.c_float), ("rope_original_max_pos", C.c_int32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class EngineConfig(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("model_name", C.c_char_p), ("preset", C.c_char_p),
                ("model", ModelConfig), ("weights_path", C.c_char_p), ("weights_seed", C.c_uint64),
                ("kv_pool_bytes", C.c_int64), ("page_size", C.c_int32), ("max_batch", C.c_int32),
                ("max_seqs", C.c_int32), ("use_cuda_graph", C.c_int32), ("decode_path", C.c_int32),
                ("start_scheduler", C.c_int32), ("reserved", C.c_int32 * 8)]


class Sampling(C.Structure):
    _fields_ = [("temperature", C.c_float), ("top_k", C.c_int32), ("top_p", C.c_float), ("repeat_penalty", C.c_float),
                ("repeat_last_n", C.c_int32), ("seed", C.c_uint64), ("max_new_tokens", C.c_int32),
                ("ignore_eos", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("text", C.c_void_p), ("text_len", C.c_size_t), ("done_reason", C.c_void_p),
                ("token_ids", C.POINTER(C.c_int32)), ("n_prompt", C.c_int32), ("n_generated", C.c_int32),
                ("prefill_ns", C.c_int64), ("decode_ns", C.c_int64), ("total_ns", C.c_int64),
                ("n_preempted", C.c_int32)]


class Logprobs(C.Structure):
    _fields_ = [("n_tokens", C.c_int32), ("top_n", C.c_int32), ("logprob", C.POINTER(C.c_float)),
                ("top_ids", C.POINTER(C.c_int32)), ("top_logprobs", C.POINTER(C.c_float))]


class Stats(C.Structure):
    _fields_ = [("tokens_per_sec", C.c_double), ("load", C.c_double), ("queue_depth", C.c_int32),
                ("active_seqs", C.c_int32), ("kv_pages_total", C.c_int32), ("kv_pages_used", C.c_int32),
                ("tokens_generated", C.c_int64), ("requests_completed", C.c_int64), ("preemptions", C.c_int64),
                ("vram_gb", C.c_int32), ("gpu_model", C.c_char * 64), ("kernel_launches", C.c_int64),
                ("measured_tokens_per_sec", C.c_double), ("sched_decode_steps", C.c_int64), ("sched_decode_ns", C.c_int64),
                ("sched_prefill_calls", C.c_int64), ("sched_prefill_tokens", C.c_int64), ("sched_prefill_ns", C.c_int64)]


# every symbol include/clengine.h declares (tests check the library exports all of them)
EXPORTS = [
    "cl_abi_version", "cl_strerror", "cl_last_error", "cl_default_engine_config", "cl_default_sampling",
    "cl_greedy_sampling", "cl_sample_token", "cl_model_preset", "cl_engine_create", "cl_engine_destroy", "cl_engine_model_config",
    "cl_engine_stats", "cl_engine_set_tensor", "cl_checkpoint_info", "cl_generate", "cl_generate_ids", "cl_generate_ids_logprobs",
    "cl_logprobs_free", "cl_generate_stream", "cl_result_free",
    "cl_handle_message", "cl_handle_message_stream", "cl_buffer_free", "cl_tokenize", "cl_detokenize", "cl_seq_create", "cl_seq_free",
    "cl_seq_len", "cl_prefill", "cl_prefill_batch", "cl_decode_step", "cl_decode_greedy", "cl_decode_greedy_batch", "cl_decode_sample_batch", "cl_decode_step_batch", "cl_seq_fake_fill",
    "cl_time_dominant_kernel", "cl_debug_kv", "cl_debug_hidden", "cl_debug_timeline",
    "cl_op_gemv", "cl_op_gemv_residual", "cl_op_rmsnorm_gemv", "cl_op_rmsnorm_gateup", "cl_op_qkv_rope_append", "cl_op_attn_decode",
    "cl_op_gemm_bf16", "cl_op_attn_prefill", "cl_op_attn_prefill_variant", "cl_op_sample", "cl_op_logprobs", "cl_op_synth_weights", "cl_kvpool_create", "cl_kvpool_destroy",
    "cl_kvpool_reserve", "cl_kvpool_release", "cl_kvpool_pages_of", "cl_kvpool_free_pages", "cl_kvpool_used_pages",
    "cl_tokenizer_load", "cl_tokenizer_free", "cl_tokenizer_encode", "cl_tokenizer_decode", "cl_tokenizer_info", "cl_engine_load_tokenizer",
]

_lib = None


# callback types of the streaming entry points (include/clengine.h: cl_token_cb, cl_frame_cb)
TOKEN_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.POINTER(C.c_int32), C.c_int32)
FRAME_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise ImportError(f"{LIB_PATH} is missing: run `python -m crowdllama_b200.build` "
                          "(there is no CPU fallback for the CUDA extension)")
    L = C.CDLL(str(LIB_PATH))
    vp, i32, i64, u64, f32, sz = C.c_void_p, C.c_int32, C.c_int64, C.c_uint64, C.c_float, C.c_size_t
    P = C.POINTER
    sig = {
        "cl_abi_version": (C.c_int, []),
        "cl_strerror": (C.c_char_p, [C.c_int]),
        "cl_last_error": (C.c_char_p, []),
        "cl_default_engine_config": (None, [P(EngineConfig)]),
        "cl_default_sampling": (None, [P(Sampling)]),
        "cl_greedy_sampling": (None, [P(Sampling), i32]),
        "cl_model_preset": (C.c_int, [C.c_char_p, P(ModelConfig)]),
        "cl_engine_create": (C.c_int, [P(EngineConfig), P(vp)]),
        "cl_engine_destroy": (None, [vp]),
        "cl_engine_model_config": (C.c_int, [vp, P(ModelConfig)]),
        "cl_engine_stats": (C.c_int, [vp, P(Stats)]),
        "cl_engine_set_tensor": (C.c_int, [vp, i32, i32, vp, i64]),
        "cl_checkpoint_info": (C.c_int, [C.c_char_p, P(ModelConfig), P(i32), P(i64)]),
        "cl_generate": (C.c_int, [vp, C.c_char_p, C.c_char_p, sz, P(Sampling), P(Result)]),
        "cl_generate_ids": (C.c_int, [vp, vp, i32, P(Sampling), P(Result)]),
        "cl_generate_ids_logprobs": (C.c_int, [vp, vp, i32, P(Sampling), i32, P(Result), P(Logprobs)]),
        "cl_logprobs_free": (None, [P(Logprobs)]),
        "cl_generate_stream": (C.c_int, [vp, C.c_char_p, C.c_char_p, sz, P(Sampling), TOKEN_CB, vp, P(Result)]),
        "cl_handle_message_stream": (C.c_int, [vp, C.c_char_p, sz, P(Sampling), FRAME_CB, vp]),
        "cl_result_free": (None, [P(Result)]),
        "cl_handle_message": (C.c_int, [vp, C.c_char_p, sz, P(Sampling), P(vp), P(sz)]),
        "cl_buffer_free": (None, [vp]),
        "cl_tokenize": (C.c_int, [vp, C.c_char_p, sz, vp, i32, P(i32)]),
        "cl_detokenize": (C.c_int, [vp, vp, i32, vp, sz, P(sz)]),
        "cl_seq_create": (C.c_int, [vp, P(i32)]),
        "cl_sample_token": (C.c_int, [vp, i32, vp, vp, i32, C.c_uint64, P(i32)]),
        "cl_seq_free": (C.c_int, [vp, i32]),
        "cl_seq_len": (C.c_int, [vp, i32, P(i32)]),
        "cl_prefill": (C.c_int, [vp, i32, vp, i32, vp]),
        "cl_prefill_batch": (C.c_int, [vp, vp, i32, vp, vp, vp]),
        "cl_decode_step": (C.c_int, [vp, i32, i32, vp, P(i32)]),
        "cl_decode_greedy": (C.c_int, [vp, i32, i32, i32, vp, P(f32)]),
        "cl_decode_greedy_batch": (C.c_int, [vp, vp, i32, vp, i32, vp, P(f32)]),
        "cl_decode_sample_batch": (C.c_int, [vp, vp, i32, vp, P(Sampling), vp, i32, vp, P(f32)]),
        "cl_decode_step_batch": (C.c_int, [vp, vp, i32, vp, vp, vp]),
        "cl_seq_fake_fill": (C.c_int, [vp, i32, i32]),
        "cl_time_dominant_kernel": (C.c_int, [vp, i32, i32, i32, P(f32), P(f32)]),
        "cl_debug_kv": (C.c_int, [vp, i32, i32, i32, i32, i32, vp]),
        "cl_debug_hidden": (C.c_int, [vp, vp, i32]),
        "cl_debug_timeline": (C.c_int, [vp, vp, i32]),
        "cl_op_gemv": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, i32, i32, i32, P(f32)]),
        "cl_op_gemv_residual": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, vp, i32, i32]),
        "cl_op_rmsnorm_gemv": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, f32, vp, i32, i32]),
        "cl_op_rmsnorm_gateup": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, f32, vp, i32, i32]),
        "cl_op_attn_decode": (C.c_int, [C.c_int, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
        "cl_op_qkv_rope_append": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, f32, i32, i32, i32, i32, i32, f32, vp, vp, vp]),
        "cl_op_gemm_bf16": (C.c_int, [C.c_int, vp, vp, vp, i32, i32, i32, i32, P(f32)]),
        "cl_op_attn_prefill": (C.c_int, [C.c_int, vp, vp, vp, i32, i32, i32, i32, vp]),
        "cl_op_attn_prefill_variant": (C.c_int, [C.c_int, C.c_int, vp, vp, vp, i32, i32, i32, i32, vp, i32, P(f32)]),
        "cl_op_sample": (C.c_int, [C.c_int, vp, i32, i32, P(Sampling), vp, vp, vp, vp, i32, P(f32)]),
        "cl_op_logprobs": (C.c_int, [C.c_int, vp, i32, i32, vp, i32, vp, vp, vp, i32, P(f32)]),
        "cl_op_synth_weights": (C.c_int, [C.c_int, u64, i32, i64, f32, vp]),
        "cl_tokenizer_load": (C.c_int, [C.c_char_p, C.c_char_p, P(vp)]),
        "cl_tokenizer_free": (None, [vp]),
        "cl_tokenizer_encode": (C.c_int, [vp, C.c_char_p, sz, i32, i32, vp, i32, P(i32)]),
        "cl_tokenizer_decode": (C.c_int, [vp, vp, i32, vp, sz, P(sz)]),
        "cl_tokenizer_info": (C.c_int, [vp, P(i32), P(i32), P(i32)]),
        "cl_engine_load_tokenizer": (C.c_int, [vp, C.c_char_p, C.c_char_p]),
        "cl_kvpool_create": (C.c_int, [i32, i32, P(vp)]),
        "cl_kvpool_destroy": (None, [vp]),
        "cl_kvpool_reserve": (C.c_int, [vp, i32, i32]),
        "cl_kvpool_release": (C.c_int, [vp, i32]),
        "cl_kvpool_pages_of": (C.c_int, [vp, i32, vp, i32, P(i32)]),
        "cl_kvpool_free_pages": (C.c_int, [vp]),
        "cl_kvpool_used_pages": (C.c_int, [vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    _lib = L
    return L


class EngineError(RuntimeError):
    def __init__(self, status: int, where: str):
        L = lib()
        self.status = status
        self.detail = L.cl_last_error().decode(errors="replace")
        super().__init__(f"{where}: {L.cl_strerror(status).decode()} ({status}) {self.detail}")


def _check(rc: int, where: str):
    if rc != CL_OK:
        raise EngineError(rc, where)


def _ptr(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def device_count() -> int:
    """Number of visible CUDA devices according to the driver (no torch involved)."""
    try:
        cuda = C.CDLL("libcuda.so.1")
    except OSError:
        return 0
    if cuda.cuInit(0) != 0:
        return 0
    n = C.c_int(0)
    if cuda.cuDeviceGetCount(C.byref(n)) != 0:
        return 0
    return n.value


def model_preset(name: str) -> dict:
    mc = ModelConfig()
    _check(lib().cl_model_preset(name.encode(), C.byref(mc)), "cl_model_preset")
    return mc.as_dict()


def checkpoint_info(path, model: dict | None = None):
    """cl_checkpoint_info: (model config, tensors, parameters) of an HF safetensors checkpoint; host-only validation."""
    mc = ModelConfig(**model) if model else ModelConfig()
    nt, npar = C.c_int32(0), C.c_int64(0)
    _check(lib().cl_checkpoint_info(str(path).encode(), C.byref(mc), C.byref(nt), C.byref(npar)), "cl_checkpoint_info")
    return mc.as_dict(), nt.value, npar.value


def greedy(max_new_tokens: int, ignore_eos: bool = False) -> Sampling:
    s = Sampling()
    lib().cl_greedy_sampling(C.byref(s), max_new_tokens)
    s.ignore_eos = 1 if ignore_eos else 0
    return s


def sample_token(logits, sampling: Sampling, history=(), step: int = 0) -> int:
    """The engine's host-side sampler on caller-provided logits (cl_sample_token; no GPU involved)."""
    lg = np.ascontiguousarray(logits, dtype=np.float32)
    h = np.ascontiguousarray(list(history), dtype=np.int32)
    out = C.c_int32()
    _check(lib().cl_sample_token(_ptr(lg), lg.size, C.byref(sampling), _ptr(h) if h.size else None, h.size, step, C.byref(out)), "cl_sample_token")
    return int(out.value)


def ollama_default_sampling(seed: int = 0, max_new_tokens: int = -1) -> Sampling:
    s = Sampling()
    lib().cl_default_sampling(C.byref(s))
    s.seed = seed
    s.max_new_tokens = max_new_tokens
    return s


class GenerateResult:
    """With log-probabilities (generate_ids(..., top_logprobs=N)): logprob [n_generated] float32, top_ids / top_logprobs
    [n_generated][N]; otherwise those three are None."""
    logprob = top_ids = top_logprobs = None

    def __init__(self, r: Result):
        self.text = C.string_at(r.text, r.text_len).decode("utf-8", errors="replace") if r.text else ""
        self.done_reason = C.string_at(r.done_reason).decode() if r.done_reason else ""
        self.token_ids = np.ctypeslib.as_array(r.token_ids, shape=(max(r.n_generated, 1),))[:r.n_generated].copy() \
            if r.n_generated else np.zeros(0, np.int32)
        self.n_prompt, self.n_generated = r.n_prompt, r.n_generated
        self.prefill_ns, self.decode_ns, self.total_ns = r.prefill_ns, r.decode_ns, r.total_ns
        self.n_preempted = r.n_preempted


class Engine:
    """One engine per GPU process (independent replicas; no NCCL on the decode path)."""

    def __init__(self, preset: str | None = None, model: dict | None = None, model_name: str | None = None,
                 device: int = 0, seed: int = 1234, max_batch: int = 8, max_seqs: int | None = None,
                 page_size: int = 32, kv_pool_bytes: int = 0, use_cuda_graph: bool = True, decode_path: int = 0,
                 start_scheduler: bool = False, weights_path: str | None = None):
        L = lib()
        cfg = EngineConfig()
        L.cl_default_engine_config(C.byref(cfg))
        cfg.device = device
        self._keep = [(model_name or preset or "model").encode(), preset.encode() if preset else None]
        cfg.model_name = self._keep[0]
        cfg.preset = self._keep[1]
        if model is not None:
            cfg.preset = None
            cfg.model = ModelConfig(**model)
        cfg.weights_seed = seed
        if weights_path is not None:
            self._keep.append(str(weights_path).encode())
            cfg.weights_path = self._keep[-1]
        cfg.max_batch = max_batch
        cfg.max_seqs = max_seqs or max_batch
        cfg.page_size = page_size
        cfg.kv_pool_bytes = kv_pool_bytes
        cfg.use_cuda_graph = 1 if use_cuda_graph else -1
        cfg.decode_path = decode_path
        cfg.start_scheduler = 1 if start_scheduler else 0
        h = C.c_void_p()
        _check(L.cl_engine_create(C.byref(cfg), C.byref(h)), "cl_engine_create")
        self._h = h
        mc = ModelConfig()
        _check(L.cl_engine_model_config(self._h, C.byref(mc)), "cl_engine_model_config")
        self.cfg = mc.as_dict()
        self.model_name = self._keep[0].decode()

    def close(self):
        if getattr(self, "_h", None):
            lib().cl_engine_destroy(self._h)
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- weights ---------------------------------------------------------------------------------
    def set_tensor(self, layer: int, kind: str, bf16: np.ndarray):
        a = np.ascontiguousarray(bf16, dtype=np.uint16)
        _check(lib().cl_engine_set_tensor(self._h, layer, KINDS[kind], _ptr(a), a.size), f"set_tensor({kind})")

    # ---- token level -----------------------------------------------------------------------------
    def seq_create(self) -> int:
        s = C.c_int32(-1)
        _check(lib().cl_seq_create(self._h, C.byref(s)), "cl_seq_create")
        return s.value

    def seq_free(self, s: int):
        _check(lib().cl_seq_free(self._h, s), "cl_seq_free")

    def seq_len(self, s: int) -> int:
        n = C.c_int32()
        _check(lib().cl_seq_len(self._h, s, C.byref(n)), "cl_seq_len")
        return n.value

    def prefill(self, s: int, ids, want_logits: bool = True):
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        out = np.empty(self.cfg["vocab_size"], np.float32) if want_logits else None
        _check(lib().cl_prefill(self._h, s, _ptr(ids), len(ids), _ptr(out) if want_logits else None), "cl_prefill")
        return out

    def prefill_batch(self, seqs, prompts, want_logits: bool = True):
        """cl_prefill_batch: several prompts in one pass; returns [n_seqs][vocab] logits of the last positions (or None)."""
        ss = np.ascontiguousarray(seqs, dtype=np.int32)
        lens = np.ascontiguousarray([len(p) for p in prompts], dtype=np.int32)
        ids = np.ascontiguousarray(np.concatenate([np.asarray(p, np.int32) for p in prompts]), dtype=np.int32)
        out = np.empty((len(ss), self.cfg["vocab_size"]), np.float32) if want_logits else None
        _check(lib().cl_prefill_batch(self._h, _ptr(ss), len(ss), _ptr(ids), _ptr(lens), _ptr(out) if want_logits else None), "cl_prefill_batch")
        return out

    def decode_step(self, s: int, tok: int, want_logits: bool = True):
        out = np.empty(self.cfg["vocab_size"], np.float32) if want_logits else None
        am = C.c_int32(-1)
        _check(lib().cl_decode_step(self._h, s, int(tok), _ptr(out) if want_logits else None, C.byref(am)),
               "cl_decode_step")
        return out, am.value

    def decode_greedy(self, s: int, first_id: int, n_steps: int):
        ids = np.empty(n_steps, np.int32)
        ms = C.c_float(0)
        _check(lib().cl_decode_greedy(self._h, s, int(first_id), n_steps, _ptr(ids), C.byref(ms)), "cl_decode_greedy")
        return ids, ms.value

    def decode_greedy_batch(self, seqs, first_ids, n_steps: int):
        seqs = np.ascontiguousarray(seqs, dtype=np.int32)
        first = np.ascontiguousarray(first_ids, dtype=np.int32)
        ids = np.empty((n_steps, len(seqs)), np.int32)
        ms = C.c_float(0)
        _check(lib().cl_decode_greedy_batch(self._h, _ptr(seqs), len(seqs), _ptr(first), n_steps, _ptr(ids),
                                            C.byref(ms)), "cl_decode_greedy_batch")
        return ids, ms.value

    def decode_sample_batch(self, seqs, first_ids, samplings, first_steps, n_steps: int):
        """cl_decode_sample_batch: n_steps batched steps, each followed by the device sampler; samplings[b] is greedy or
        within the device limits.  Returns (ids [n_steps][B], device ms)."""
        seqs = np.ascontiguousarray(seqs, dtype=np.int32)
        first = np.ascontiguousarray(first_ids, dtype=np.int32)
        sps = (Sampling * len(seqs))(*samplings)
        steps = np.ascontiguousarray(first_steps, dtype=np.uint64)
        ids = np.empty((n_steps, len(seqs)), np.int32)
        ms = C.c_float(0)
        _check(lib().cl_decode_sample_batch(self._h, _ptr(seqs), len(seqs), _ptr(first), sps, _ptr(steps), n_steps, _ptr(ids),
                                            C.byref(ms)), "cl_decode_sample_batch")
        return ids, ms.value

    def decode_step_batch(self, seqs, toks, want_logits: bool = True):
        """One batched step with caller-chosen tokens; returns (logits [B][V] or None, greedy next ids [B])."""
        seqs = np.ascontiguousarray(seqs, dtype=np.int32)
        toks = np.ascontiguousarray(toks, dtype=np.int32)
        out = np.empty((len(seqs), self.cfg["vocab_size"]), np.float32) if want_logits else None
        am = np.empty(len(seqs), np.int32)
        _check(lib().cl_decode_step_batch(self._h, _ptr(seqs), len(seqs), _ptr(toks), _ptr(out) if want_logits else None, _ptr(am)),
               "cl_decode_step_batch")
        return out, am

    def seq_fake_fill(self, s: int, n_tokens: int):
        """Fill the sequence's paged KV (all layers) with the synthetic cache pattern the parity tests' CPU checker also
        generates (include/clengine.h: cl_seq_fake_fill) — a parity aid."""
        _check(lib().cl_seq_fake_fill(self._h, s, n_tokens), "cl_seq_fake_fill")

    def debug_kv(self, s: int, layer: int, which: int, t0: int, n: int) -> np.ndarray:
        """Cached K (which=0) / V (which=1) rows of `layer` for tokens t0..t0+n-1: [n][n_kv*head_dim] fp32."""
        out = np.empty((n, self.cfg["n_kv_heads"] * self.cfg["head_dim"]), np.float32)
        _check(lib().cl_debug_kv(self._h, s, layer, which, t0, n, _ptr(out)), "cl_debug_kv")
        return out

    def time_dominant_kernel(self, s: int, first_id: int, n_steps: int):
        """(kernel_ms, step_ms): mean CUDA-event time of the dominant kernel / of the whole eagerly launched step."""
        k, t = C.c_float(0), C.c_float(0)
        _check(lib().cl_time_dominant_kernel(self._h, s, int(first_id), n_steps, C.byref(k), C.byref(t)), "cl_time_dominant_kernel")
        return k.value, t.value

    def debug_hidden(self) -> np.ndarray:
        out = np.empty(self.cfg["d_model"], np.float32)
        _check(lib().cl_debug_hidden(self._h, _ptr(out), out.size), "cl_debug_hidden")
        return out

    def debug_timeline(self) -> np.ndarray:
        n = (self.cfg["n_layers"] * 5 + 1) * 4
        out = np.zeros(n, np.int64)
        rc = lib().cl_debug_timeline(self._h, _ptr(out), n)
        if rc < 0:
            raise EngineError(rc, "cl_debug_timeline")
        return out.reshape(-1, 4)

    # ---- request level ---------------------------------------------------------------------------
    def generate_ids(self, prompt_ids, sampling: Sampling, top_logprobs: int | None = None) -> GenerateResult:
        """top_logprobs (0..MAX_TOP_LOGPROBS): also return the log-probability of every generated token with that many
        alternatives (cl_generate_ids_logprobs); None: cl_generate_ids."""
        ids = np.ascontiguousarray(prompt_ids, dtype=np.int32)
        r = Result()
        if top_logprobs is None:
            _check(lib().cl_generate_ids(self._h, _ptr(ids), len(ids), C.byref(sampling), C.byref(r)), "cl_generate_ids")
            try:
                return GenerateResult(r)
            finally:
                lib().cl_result_free(C.byref(r))
        lp = Logprobs()
        _check(lib().cl_generate_ids_logprobs(self._h, _ptr(ids), len(ids), C.byref(sampling), int(top_logprobs), C.byref(r), C.byref(lp)),
               "cl_generate_ids_logprobs")
        try:
            g = GenerateResult(r)
            n, k = lp.n_tokens, lp.top_n
            g.logprob = np.ctypeslib.as_array(lp.logprob, shape=(n,)).copy() if n else np.zeros(0, np.float32)
            if k and n:
                g.top_ids = np.ctypeslib.as_array(lp.top_ids, shape=(n * k,)).reshape(n, k).copy()
                g.top_logprobs = np.ctypeslib.as_array(lp.top_logprobs, shape=(n * k,)).reshape(n, k).copy()
            else:
                g.top_ids, g.top_logprobs = np.zeros((n, k), np.int32), np.zeros((n, k), np.float32)
            return g
        finally:
            lib().cl_result_free(C.byref(r))
            lib().cl_logprobs_free(C.byref(lp))

    def generate(self, model: str, prompt: str, sampling: Sampling | None = None) -> GenerateResult:
        r = Result()
        p = prompt.encode("utf-8")
        _check(lib().cl_generate(self._h, model.encode(), p, len(p), C.byref(sampling) if sampling else None,
                                 C.byref(r)), "cl_generate")
        try:
            return GenerateResult(r)
        finally:
            lib().cl_result_free(C.byref(r))

    def generate_stream(self, model: str, prompt: str, sampling: Sampling | None = None, on_text=None) -> GenerateResult:
        """cl_generate_stream: on_text(text_delta: str, ids: list[int]) is called on this thread as tokens arrive;
        a truthy return cancels the request."""
        r = Result()
        p = prompt.encode("utf-8")

        def cb(user, text, text_len, ids, n_ids):
            try:
                delta = C.string_at(text, text_len).decode("utf-8", "replace") if text_len else ""
                new = [ids[i] for i in range(n_ids)] if n_ids else []
                return 1 if (on_text and on_text(delta, new)) else 0
            except Exception:       # never unwind through the C frames
                return 1

        cfn = TOKEN_CB(cb)
        _check(lib().cl_generate_stream(self._h, model.encode(), p, len(p), C.byref(sampling) if sampling else None, cfn, None,
                                        C.byref(r)), "cl_generate_stream")
        try:
            return GenerateResult(r)
        finally:
            lib().cl_result_free(C.byref(r))

    def handle_message_stream(self, req: bytes, sampling: Sampling | None = None, on_frame=None) -> int:
        """cl_handle_message_stream: on_frame(serialised BaseMessage) per response frame; returns the frame count."""
        n = [0]

        def cb(user, msg, length):
            try:
                n[0] += 1
                return 1 if (on_frame and on_frame(C.string_at(msg, length))) else 0
            except Exception:
                return 1

        cfn = FRAME_CB(cb)
        _check(lib().cl_handle_message_stream(self._h, req, len(req), C.byref(sampling) if sampling else None, cfn, None),
               "cl_handle_message_stream")
        return n[0]

    def handle_message(self, req: bytes, sampling: Sampling | None = None) -> bytes:
        out, n = C.c_void_p(), C.c_size_t()
        _check(lib().cl_handle_message(self._h, req, len(req), C.byref(sampling) if sampling else None,
                                       C.byref(out), C.byref(n)), "cl_handle_message")
        try:
            return C.string_at(out, n.value)
        finally:
            lib().cl_buffer_free(out)

    def load_tokenizer(self, tokenizer_json_path: str, chat_family: str | None = None) -> None:
        """Replace the byte-level fallback by an HF tokenizer.json (cl_engine_load_tokenizer)."""
        _check(lib().cl_engine_load_tokenizer(self._h, str(tokenizer_json_path).encode(), chat_family.encode() if chat_family else None),
               "cl_engine_load_tokenizer")

    def tokenize(self, text: str) -> np.ndarray:
        b = text.encode("utf-8")
        n = C.c_int32()
        _check(lib().cl_tokenize(self._h, b, len(b), None, 0, C.byref(n)), "cl_tokenize")
        ids = np.empty(n.value, np.int32)
        _check(lib().cl_tokenize(self._h, b, len(b), _ptr(ids), n.value, C.byref(n)), "cl_tokenize")
        return ids

    def detokenize(self, ids) -> str:
        ids = np.ascontiguousarray(ids, dtype=np.int32)
        n = C.c_size_t()
        _check(lib().cl_detokenize(self._h, _ptr(ids), len(ids), None, 0, C.byref(n)), "cl_detokenize")
        buf = C.create_string_buffer(n.value + 1)
        _check(lib().cl_detokenize(self._h, _ptr(ids), len(ids), buf, n.value + 1, C.byref(n)), "cl_detokenize")
        return buf.value.decode("utf-8", errors="replace")

    def stats(self) -> dict:
        st = Stats()
        _check(lib().cl_engine_stats(self._h, C.byref(st)), "cl_engine_stats")
        d = {n: getattr(st, n) for n, _ in st._fields_}
        d["gpu_model"] = st.gpu_model.decode(errors="replace")
        return d


# ---- single-op wrappers (host numpy in / out) -----------------------------------------------------
def op_gemv(w_bf16, x, variant=0, iters=0, device=0):
    w = np.ascontiguousarray(w_bf16, dtype=np.uint16)
    x = np.ascontiguousarray(x, dtype=np.float32)
    y = np.empty(w.shape[0], np.float32)
    ms = C.c_float(0)
    _check(lib().cl_op_gemv(device, variant, _ptr(w), _ptr(x), _ptr(y), w.shape[0], w.shape[1], iters, C.byref(ms)),
           "cl_op_gemv")
    return (y, ms.value) if iters else y


def op_gemv_residual(w_bf16, x, resid, variant=0, device=0):
    w = np.ascontiguousarray(w_bf16, dtype=np.uint16)
    x = np.ascontiguousarray(x, dtype=np.float32)
    r = np.ascontiguousarray(resid, dtype=np.float32)
    y = np.empty(w.shape[0], np.float32)
    _check(lib().cl_op_gemv_residual(device, variant, _ptr(w), _ptr(x), _ptr(r), _ptr(y), w.shape[0], w.shape[1]),
           "cl_op_gemv_residual")
    return y


def op_rmsnorm_gemv(w_bf16, h, gain, eps, variant=0, device=0):
    w = np.ascontiguousarray(w_bf16, dtype=np.uint16)
    h = np.ascontiguousarray(h, dtype=np.float32)
    g = np.ascontiguousarray(gain, dtype=np.float32)
    y = np.empty(w.shape[0], np.float32)
    _check(lib().cl_op_rmsnorm_gemv(device, variant, _ptr(w), _ptr(h), _ptr(g), eps, _ptr(y), w.shape[0], w.shape[1]),
           "cl_op_rmsnorm_gemv")
    return y


def op_rmsnorm_gateup(w_gu_bf16, h, gain, eps, variant=0, device=0):
    w = np.ascontiguousarray(w_gu_bf16, dtype=np.uint16)
    h = np.ascontiguousarray(h, dtype=np.float32)
    g = np.ascontiguousarray(gain, dtype=np.float32)
    act = np.empty(w.shape[0] // 2, np.float32)
    _check(lib().cl_op_rmsnorm_gateup(device, variant, _ptr(w), _ptr(h), _ptr(g), eps, _ptr(act), w.shape[0] // 2,
                                      w.shape[1]), "cl_op_rmsnorm_gateup")
    return act


def op_attn_decode(q_roped, k_cache_bf16, v_cache_bf16, n_heads, n_kv, head_dim, page_size=32, device=0):
    q = np.ascontiguousarray(q_roped, dtype=np.float32)
    kc = np.ascontiguousarray(k_cache_bf16, dtype=np.uint16)
    vc = np.ascontiguousarray(v_cache_bf16, dtype=np.uint16)
    out = np.empty(n_heads * head_dim, np.float32)
    _check(lib().cl_op_attn_decode(device, _ptr(q), _ptr(kc), _ptr(vc), kc.shape[0], n_heads, n_kv, head_dim, page_size,
                                   _ptr(out)), "cl_op_attn_decode")
    return out


def op_qkv_rope_append(w_qkv_bf16, h, gain, eps, n_heads, n_kv, head_dim, pos, rope_theta, variant=0, device=0):
    w = np.ascontiguousarray(w_qkv_bf16, dtype=np.uint16)
    h = np.ascontiguousarray(h, dtype=np.float32)
    g = np.ascontiguousarray(gain, dtype=np.float32)
    q = np.empty(n_heads * head_dim, np.float32)
    k = np.empty(n_kv * head_dim, np.uint16)
    v = np.empty(n_kv * head_dim, np.uint16)
    _check(lib().cl_op_qkv_rope_append(device, variant, _ptr(w), _ptr(h), _ptr(g), eps, w.shape[1], n_heads, n_kv, head_dim, pos,
                                       rope_theta, _ptr(q), _ptr(k), _ptr(v)), "cl_op_qkv_rope_append")
    return q, k, v


def op_gemm_bf16(x_bf16, w_bf16, iters=0, device=0):
    x = np.ascontiguousarray(x_bf16, dtype=np.uint16)
    w = np.ascontiguousarray(w_bf16, dtype=np.uint16)
    y = np.empty((x.shape[0], w.shape[0]), np.float32)
    ms = C.c_float(0)
    _check(lib().cl_op_gemm_bf16(device, _ptr(x), _ptr(w), _ptr(y), x.shape[0], w.shape[0], w.shape[1], iters,
                                 C.byref(ms)), "cl_op_gemm_bf16")
    return (y, ms.value) if iters else y


def op_attn_prefill(q_bf16, k_bf16, v_bf16, n_heads, n_kv, head_dim, device=0):
    q = np.ascontiguousarray(q_bf16, dtype=np.uint16)
    k = np.ascontiguousarray(k_bf16, dtype=np.uint16)
    v = np.ascontiguousarray(v_bf16, dtype=np.uint16)
    t = q.shape[0]
    out = np.empty((t, n_heads * head_dim), np.float32)
    _check(lib().cl_op_attn_prefill(device, _ptr(q), _ptr(k), _ptr(v), t, n_heads, n_kv, head_dim, _ptr(out)),
           "cl_op_attn_prefill")
    return out


def op_attn_prefill_variant(q_bf16, k_bf16, v_bf16, n_heads, n_kv, head_dim, variant, iters=0, device=0):
    """variant 0: mma.sync kernel, 1: tcgen05 kernel, -1: auto.  Returns (out, ms per launch or None)."""
    q = np.ascontiguousarray(q_bf16, dtype=np.uint16)
    k = np.ascontiguousarray(k_bf16, dtype=np.uint16)
    v = np.ascontiguousarray(v_bf16, dtype=np.uint16)
    t = q.shape[0]
    out = np.empty((t, n_heads * head_dim), np.float32)
    ms = C.c_float(0)
    _check(lib().cl_op_attn_prefill_variant(device, variant, _ptr(q), _ptr(k), _ptr(v), t, n_heads, n_kv, head_dim, _ptr(out), iters,
                                            C.byref(ms)), "cl_op_attn_prefill_variant")
    return out, (ms.value if iters > 0 else None)


def op_sample(logits, samplings, windows, steps, iters=0, device=0):
    """cl_op_sample: the device sampler on host logits [n_rows][vocab]; windows[r] = row r's history (at most
    SAMPLE_MAX_WINDOW ids).  Returns (ids [n_rows], mean ms of `iters` timed launches or 0)."""
    lg = np.ascontiguousarray(logits, dtype=np.float32)
    n, v = lg.shape
    win = np.zeros((n, SAMPLE_MAX_WINDOW), np.int32)
    nwin = np.zeros(n, np.int32)
    for r, w in enumerate(windows):
        w = np.asarray(w, np.int32)
        if w.size > SAMPLE_MAX_WINDOW:
            raise ValueError(f"window of row {r} holds {w.size} ids (at most {SAMPLE_MAX_WINDOW})")
        win[r, :w.size] = w
        nwin[r] = w.size
    sps = (Sampling * n)(*samplings)
    st = np.ascontiguousarray(steps, dtype=np.uint64)
    ids = np.empty(n, np.int32)
    ms = C.c_float(0)
    _check(lib().cl_op_sample(device, _ptr(lg), n, v, sps, _ptr(win), _ptr(nwin), _ptr(st), _ptr(ids), iters, C.byref(ms)),
           "cl_op_sample")
    return ids, ms.value


def op_logprobs(logits, chosen, top_n, iters=0, device=0):
    """cl_op_logprobs: logprobs_kernel on host logits [n_rows][vocab] with chosen[n_rows] the emitted ids.  Returns
    (logprob [n_rows], top_ids [n_rows][top_n], top_logprobs [n_rows][top_n], mean ms of `iters` timed launches or 0)."""
    lg = np.ascontiguousarray(logits, dtype=np.float32)
    n, v = lg.shape
    ch = np.ascontiguousarray(chosen, dtype=np.int32)
    if ch.shape != (n,):
        raise ValueError("chosen needs one id per row")
    lp = np.empty(n, np.float32)
    ids = np.empty((n, max(top_n, 0)), np.int32)
    tl = np.empty((n, max(top_n, 0)), np.float32)
    ms = C.c_float(0)
    _check(lib().cl_op_logprobs(device, _ptr(lg), n, v, _ptr(ch), int(top_n), _ptr(lp), _ptr(ids) if top_n > 0 else None,
                                _ptr(tl) if top_n > 0 else None, iters, C.byref(ms)), "cl_op_logprobs")
    return lp, ids, tl, ms.value


def op_synth_weights(seed, key, n, scale, device=0):
    out = np.empty(n, np.uint16)
    _check(lib().cl_op_synth_weights(device, seed, key, n, scale, _ptr(out)), "cl_op_synth_weights")
    return out


class HfTokenizer:
    """Native tokenizer.json loader (csrc/tokenizer.cpp) — host logic, works without a GPU."""

    def __init__(self, tokenizer_json_path, chat_family: str | None = None):
        h = C.c_void_p()
        _check(lib().cl_tokenizer_load(str(tokenizer_json_path).encode(), chat_family.encode() if chat_family else None, C.byref(h)),
               "cl_tokenizer_load")
        self._h = h
        v, b, e = C.c_int32(), C.c_int32(), C.c_int32()
        _check(lib().cl_tokenizer_info(self._h, C.byref(v), C.byref(b), C.byref(e)), "cl_tokenizer_info")
        self.vocab_size, self.bos, self.eos = v.value, b.value, e.value

    def encode(self, text: str, add_bos: bool = False, chat: bool = False) -> list:
        b = text.encode("utf-8")
        n = C.c_int32()
        _check(lib().cl_tokenizer_encode(self._h, b, len(b), int(add_bos), int(chat), None, 0, C.byref(n)), "cl_tokenizer_encode")
        ids = np.zeros(max(n.value, 1), np.int32)
        _check(lib().cl_tokenizer_encode(self._h, b, len(b), int(add_bos), int(chat), _ptr(ids), n.value, C.byref(n)), "cl_tokenizer_encode")
        return ids[:n.value].tolist()

    def decode(self, ids) -> str:
        a = np.ascontiguousarray(ids, dtype=np.int32)
        n = C.c_size_t()
        _check(lib().cl_tokenizer_decode(self._h, _ptr(a), len(a), None, 0, C.byref(n)), "cl_tokenizer_decode")
        buf = C.create_string_buffer(n.value + 1)
        _check(lib().cl_tokenizer_decode(self._h, _ptr(a), len(a), buf, n.value, C.byref(n)), "cl_tokenizer_decode")
        return buf.raw[:n.value].decode("utf-8", errors="replace")

    def close(self):
        if getattr(self, "_h", None):
            lib().cl_tokenizer_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class KvPool:
    """Host-side paged-KV allocator (usable without a GPU)."""

    def __init__(self, n_pages: int, page_size: int):
        h = C.c_void_p()
        _check(lib().cl_kvpool_create(n_pages, page_size, C.byref(h)), "cl_kvpool_create")
        self._h = h

    def close(self):
        if self._h:
            lib().cl_kvpool_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reserve(self, owner: int, n_tokens: int) -> int:
        return lib().cl_kvpool_reserve(self._h, owner, n_tokens)

    def release(self, owner: int) -> int:
        return lib().cl_kvpool_release(self._h, owner)

    def pages_of(self, owner: int):
        n = C.c_int32()
        lib().cl_kvpool_pages_of(self._h, owner, None, 0, C.byref(n))
        a = np.empty(max(n.value, 1), np.int32)
        _check(lib().cl_kvpool_pages_of(self._h, owner, _ptr(a), a.size, C.byref(n)), "cl_kvpool_pages_of")
        return a[:n.value].tolist()

    @property
    def free_pages(self) -> int:
        return lib().cl_kvpool_free_pages(self._h)

    @property
    def used_pages(self) -> int:
        return lib().cl_kvpool_used_pages(self._h)
