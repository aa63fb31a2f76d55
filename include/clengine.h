/*
 * clengine.h — C-ABI of the B200-native CrowdLlama worker decode engine (libclengine.so).
 *
 * This is the drop-in boundary for the ONE hot path this repository accelerates: the
 * worker-side model step that the reference reaches through
 *     crowdllama.UnifiedAPIHandler            /root/reference/pkg/crowdllama/api.go:19
 *     crowdllama.WorkerAPIHandler             /root/reference/pkg/crowdllama/api.go:45-96
 *     callOllamaAPI (HTTP POST /api/chat)     /root/reference/pkg/crowdllama/api.go:108-160
 * and, behind that HTTP call, the un-vendored github.com/ollama/ollama v0.9.6
 * (/root/reference/go.mod:12) llama.cpp decode loop.  A Go cgo shim (go/b200handler/handler.go,
 * shown in INTEGRATION.md) builds a UnifiedAPIHandler closure over cl_generate(); Python tests
 * and bench.py bind the same symbols with ctypes.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no C++/torch types.
 *   - every function returns 0 (CL_OK) or a negative cl_status; nothing throws across the ABI.
 *   - the library never retains caller pointers after a call returns (cgo rule); strings and
 *     id arrays handed back in cl_result are malloc()'d by the library and released with
 *     cl_result_free().
 *   - cl_generate(), cl_generate_ids(), cl_engine_stats() are thread-safe and re-entrant (one goroutine per inbound
 *     libp2p stream calls the handler concurrently: /root/reference/pkg/peer/peer.go:177-182).
 *     The token-level cl_seq_* / cl_prefill / cl_decode_step calls are serialised internally by one engine lock.
 *   - there is NO CPU fallback: if no sm_100 device is present cl_engine_create fails with
 *     CL_ERR_NO_DEVICE.
 */
#ifndef CLENGINE_H_
#define CLENGINE_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CL_ABI_VERSION 2

typedef enum cl_status {
  CL_OK = 0,
  CL_ERR_INVALID_ARG = -1,
  CL_ERR_NO_DEVICE = -2,     /* no CUDA device / not sm_100 */
  CL_ERR_CUDA = -3,          /* CUDA runtime error; see cl_last_error() */
  CL_ERR_OOM = -4,           /* device memory or KV pages exhausted */
  CL_ERR_UNKNOWN_MODEL = -5, /* model name not served by this engine */
  CL_ERR_TOO_LONG = -6,      /* prompt + generation exceeds max_seq_len */
  CL_ERR_BAD_SEQ = -7,       /* unknown / freed sequence handle */
  CL_ERR_SHUTDOWN = -8,      /* engine is being destroyed */
  CL_ERR_IO = -9,            /* weight / tokenizer file error */
  CL_ERR_INTERNAL = -10,
  CL_ERR_BAD_MESSAGE = -11   /* cl_handle_message: not a GenerateRequest (api.go:48-51) */
} cl_status;

/* Llama-family architecture description (public architecture facts; SURVEY.md §8). */
typedef struct cl_model_config {
  int32_t n_layers;
  int32_t d_model;
  int32_t n_heads;
  int32_t n_kv_heads;
  int32_t head_dim;
  int32_t d_ff;
  int32_t vocab_size;
  int32_t max_seq_len;   /* positions covered by the RoPE table and block tables */
  float rope_theta;
  float rms_eps;
  /* "llama3" rotary scaling (Llama-3.1 / 3.2 checkpoints; HF config.json rope_scaling / rope_parameters with
   * rope_type "llama3").  rope_factor <= 1 (e.g. 0): plain rotary embeddings.  Otherwise the inverse frequency of
   * dimension pair i is divided by rope_factor where its wavelength exceeds rope_original_max_pos / rope_low_freq_factor,
   * kept where it is below rope_original_max_pos / rope_high_freq_factor, and blended linearly in between. */
  float rope_factor;
  float rope_low_freq_factor;
  float rope_high_freq_factor;
  int32_t rope_original_max_pos;
} cl_model_config;

typedef struct cl_engine_config {
  int32_t abi_version;     /* must be CL_ABI_VERSION */
  int32_t device;          /* CUDA ordinal (one engine process per GPU) */
  const char* model_name;  /* name advertised / matched exactly, like Resource.SupportedModels
                              (/root/reference/pkg/peermanager/manager.go:349-354) */
  const char* preset;      /* "llama3-8b" | "mistral-7b" | "tinyllama-1.1b" | "tiny-test" | NULL
                              (NULL => take `model` below) */
  cl_model_config model;   /* used when preset == NULL */
  const char* weights_path;/* HF llama-layout checkpoint: a .safetensors file, or a model directory with *.safetensors shards
                              (+ config.json, used when preset == NULL and model.n_layers == 0, + tokenizer.json, loaded
                              when present); BF16 / F16 / F32 tensors -> bf16.  NULL => synthetic seeded weights */
  uint64_t weights_seed;   /* seed of the counter-based synthetic weight generator */
  int64_t kv_pool_bytes;   /* bytes of HBM for the paged KV pool; 0 => derive from max_seqs */
  int32_t page_size;       /* tokens per KV page: 16, 32 or 64 (0 => 32) */
  int32_t max_batch;       /* max concurrently decoding sequences (0 => 8); the tensor-core batched step serves 2..128,
                              larger values fall back to per-sequence GEMV kernels */
  int32_t max_seqs;        /* max live sequence handles (0 => max_batch) */
  int32_t use_cuda_graph;  /* 1 => capture the token step in a CUDA graph (default 1; -1 => 0) */
  int32_t decode_path;     /* 0 auto, 1 = generic LDG GEMV kernels, 2 = TMA-ring streaming GEMV */
  int32_t start_scheduler; /* 1 => start the continuous-batching thread behind cl_generate */
  int32_t reserved[8];
} cl_engine_config;

/* Sampler.  The reference sends no options (api.go:109-118), so Ollama defaults apply upstream:
 * temperature 0.8, top_k 40, top_p 0.9, repeat_penalty 1.1 over the last 64 tokens, random seed.
 * temperature <= 0 selects greedy argmax with lowest-index tie-break (the parity mode). */
typedef struct cl_sampling {
  float temperature;
  int32_t top_k;
  float top_p;
  float repeat_penalty;
  int32_t repeat_last_n;
  uint64_t seed;
  int32_t max_new_tokens;  /* num_predict; <= 0 => until EOS or context full */
  int32_t ignore_eos;      /* 1 => never stop on EOS (benchmarks) */
} cl_sampling;

/* Device sampler limits.  A sampled request is drawn on the GPU (no logits copy to the host) when temperature > 0,
 * 1 <= top_k <= CL_SAMPLE_MAX_TOP_K, top_k < vocab_size, and the repeat penalty is off (repeat_penalty == 1 or
 * repeat_last_n == 0) or 0 < repeat_last_n <= CL_SAMPLE_MAX_WINDOW.  Every other request is sampled on the host by
 * cl_sample_token; both draw the same token from the same logits, history and step. */
#define CL_SAMPLE_MAX_TOP_K 128
#define CL_SAMPLE_MAX_WINDOW 64

/* Log-probabilities of the generated tokens (Ollama `logprobs` / `top_logprobs`).  The numbers describe the model's raw
 * next-token distribution, log_softmax of the fp32 logits of the step, before the repeat penalty, the temperature and
 * the top-k / top-p cuts; they are the same for greedy and sampled requests.  For generated token i:
 *   logprob[i]                          = logits[token_ids[i]] - logsumexp(logits)
 *   top_ids[i * top_n + j], top_logprobs[i * top_n + j], j < top_n
 *                                       = the top_n most likely ids, value descending, then id ascending
 * Computed on the device (logprobs_kernel), one launch per step over the rows that asked; bit-reproducible. */
#define CL_MAX_TOP_LOGPROBS 20
typedef struct cl_logprobs {
  int32_t n_tokens;        /* == cl_result.n_generated */
  int32_t top_n;
  float* logprob;          /* [n_tokens], malloc'd */
  int32_t* top_ids;        /* [n_tokens][top_n], malloc'd (NULL when top_n == 0) */
  float* top_logprobs;     /* [n_tokens][top_n], malloc'd (NULL when top_n == 0) */
} cl_logprobs;
void cl_logprobs_free(cl_logprobs* l);

typedef struct cl_result {
  char* text;            /* NUL-terminated UTF-8, malloc'd */
  size_t text_len;
  char* done_reason;     /* "stop" | "length", malloc'd (GenerateResponse.DoneReason, api.go:82) */
  int32_t* token_ids;    /* generated ids, malloc'd */
  int32_t n_prompt;
  int32_t n_generated;
  int64_t prefill_ns;
  int64_t decode_ns;
  int64_t total_ns;
  int32_t n_preempted;   /* times this request was evicted and recomputed */
} cl_result;

typedef struct cl_stats {
  double tokens_per_sec;     /* capacity, load-independent: 70 % of the HBM roofline of one decode step x max_batch, from the
                                device's memory bandwidth and the model's bytes per token -> Resource.TokensThroughput (types.go:33) */
  double load;               /* (active + queued) / max_batch; > 1: requests are waiting for a batch slot -> Resource.Load
                                (types.go:35) through the two-level rule of INTEGRATION.md "What to advertise" */
  int32_t queue_depth;
  int32_t active_seqs;
  int32_t kv_pages_total;
  int32_t kv_pages_used;
  int64_t tokens_generated;
  int64_t requests_completed;
  int64_t preemptions;
  int32_t vram_gb;           /* -> Resource.VRAMGB */
  char gpu_model[64];        /* -> Resource.GPUModel */
  int64_t kernel_launches;   /* kernels of this library launched so far (graph nodes counted) */
  double measured_tokens_per_sec; /* EWMA of decode steps/s x max_batch at the CURRENT batch sizes (diagnostic; not for routing) */
  /* scheduler accounting since engine creation: batched decode steps (tokens_generated / sched_decode_steps = mean batch)
     and admission-time prefill calls, with the scheduler thread's wall time inside each */
  int64_t sched_decode_steps, sched_decode_ns;
  int64_t sched_prefill_calls, sched_prefill_tokens, sched_prefill_ns;
} cl_stats;

typedef struct cl_engine cl_engine;
typedef int32_t cl_seq_t;

/* ---- lifecycle -------------------------------------------------------------------------- */
int cl_abi_version(void);
const char* cl_strerror(int status);
/* thread-local description of the last failing call on this thread ("" if none) */
const char* cl_last_error(void);
void cl_default_engine_config(cl_engine_config* cfg);
void cl_default_sampling(cl_sampling* s);        /* Ollama defaults listed above */
void cl_greedy_sampling(cl_sampling* s, int32_t max_new_tokens);
/* The engine's host-side sampler on caller-provided logits (no GPU involved): repeat penalty over the last repeat_last_n
 * ids of `history` -> top-k -> softmax at `temperature` -> top-p -> one draw from the counter-based generator at
 * (seed, step).  Exposed so that each stage can be checked against an independent implementation
 * (tests/test_host_logic.py pins it to the HF transformers logits processors). */
int cl_sample_token(const float* logits, int32_t vocab, const cl_sampling* s, const int32_t* history, int32_t n_history,
                    uint64_t step, int32_t* id);
int cl_model_preset(const char* name, cl_model_config* out);

/* replaces: embedded Ollama server start, /root/reference/cmd/crowdllama/main.go:283-297 */
int cl_engine_create(const cl_engine_config* cfg, cl_engine** out);
void cl_engine_destroy(cl_engine* e);
int cl_engine_model_config(const cl_engine* e, cl_model_config* out);
int cl_engine_stats(cl_engine* e, cl_stats* out);
/* Overwrite one weight tensor from host memory (bf16 bits, logical [out][in] row-major; norm
 * gains as bf16 too).  kind: 0 embed, 1 lm_head, 2 final_norm, 3 attn_norm, 4 wq, 5 wk, 6 wv,
 * 7 wo, 8 ffn_norm, 9 w_gate, 10 w_up, 11 w_down (same numbering as the synthetic generator).
 * Used to load real checkpoints tensor by tensor and by the HF golden-vector parity tests. */
int cl_engine_set_tensor(cl_engine* e, int32_t layer, int32_t kind, const uint16_t* data, int64_t n);

/* Host-only check of a checkpoint (no GPU needed): parses config.json (when cfg_io->n_layers == 0 and path is a model
 * directory; the result is written back) and every safetensors header, validating tensor names, dtypes, shapes and
 * offsets against the architecture exactly as cl_engine_create does.  n_tensors / n_params (may be NULL): what the
 * engine would load. */
int cl_checkpoint_info(const char* path, cl_model_config* cfg_io, int32_t* n_tensors, int64_t* n_params);

/* ---- request level (what the Go shim calls) --------------------------------------------- */
/* replaces: callOllamaAPI, api.go:108-160.  Blocking; enqueues into the continuous-batching
 * scheduler.  `model` must equal the engine's model_name (else CL_ERR_UNKNOWN_MODEL).  The
 * prompt is raw user text (api.go:111-116 forces role "user"); it is copied before return. */
int cl_generate(cl_engine* e, const char* model, const char* prompt, size_t prompt_len,
                const cl_sampling* s, cl_result* out);
/* token-id variant of the same path (tokenizer bypass; used by parity tests and bench.py) */
int cl_generate_ids(cl_engine* e, const int32_t* prompt_ids, int32_t n_prompt,
                    const cl_sampling* s, cl_result* out);
void cl_result_free(cl_result* r);
/* cl_generate_ids with the log-probabilities of every generated token (CL_MAX_TOP_LOGPROBS above): lp receives one
 * entry per id of out->token_ids, each with its top_n (0..CL_MAX_TOP_LOGPROBS, else CL_ERR_INVALID_ARG) most likely
 * alternatives; free it with cl_logprobs_free.  The ids are the ones cl_generate_ids returns for the same request. */
int cl_generate_ids_logprobs(cl_engine* e, const int32_t* prompt_ids, int32_t n_prompt, const cl_sampling* s,
                             int32_t top_n, cl_result* out, cl_logprobs* lp);

/* Streaming variant of cl_generate (SURVEY.md §8f row 4; the reference rejects stream:true, api.go:155).
 * cb runs on the CALLING thread (cgo-safe) with each batch of new tokens: text = UTF-8 delta that later tokens
 * cannot change (an incomplete multi-byte tail is held back), ids/n_ids = the new token ids (NULL/0 for the final
 * flush).  A nonzero return cancels the request (done_reason "cancelled").  out receives the whole result. */
typedef int (*cl_token_cb)(void* user, const char* text, size_t text_len, const int32_t* ids, int32_t n_ids);
int cl_generate_stream(cl_engine* e, const char* model, const char* prompt, size_t prompt_len,
                       const cl_sampling* s, cl_token_cb cb, void* user, cl_result* out);
/* Byte-level streaming handler: like cl_handle_message, but when GenerateRequest.stream is set the answer is a
 * sequence of serialised BaseMessage{GenerateResponse} frames — Done=false frames carrying text deltas, then one
 * Done=true frame with done_reason — each handed to cb (the host writes them length-prefixed to the stream,
 * pbwire.go:14-33).  Without stream: exactly one Done=true frame.  GenerateRequest.options (field 4, the proto
 * extension of §8f row 3: seed, temperature, top_k, top_p, repeat_penalty, repeat_last_n, num_predict, raw)
 * override `s` field by field in both entry points.  With options.logprobs (field 9) every GenerateResponse carries
 * GenerateResponse.logprobs (field 8): one TokenLogprob per token id the frame covers, with options.top_logprobs
 * (field 10, 0..CL_MAX_TOP_LOGPROBS, else CL_ERR_INVALID_ARG) alternatives each. */
typedef int (*cl_frame_cb)(void* user, const uint8_t* msg, size_t len);
int cl_handle_message_stream(cl_engine* e, const uint8_t* req, size_t req_len, const cl_sampling* s,
                             cl_frame_cb cb, void* user);
/* replaces: WorkerAPIHandler, api.go:45-96, at the byte level.  `req`/`req_len` is a serialised
 * llama.v1.BaseMessage (the payload pbwire.go:14-41 length-prefixes); on success *resp is a
 * malloc'd serialised BaseMessage{GenerateResponse} (free with cl_buffer_free).  A request that
 * is not a GenerateRequest returns CL_ERR_BAD_MESSAGE (api.go:48-51). */
int cl_handle_message(cl_engine* e, const uint8_t* req, size_t req_len, const cl_sampling* s,
                      uint8_t** resp, size_t* resp_len);
void cl_buffer_free(void* p);

/* tokenizer of the served model (byte-level fallback when no vocab file is configured) */
int cl_tokenize(cl_engine* e, const char* text, size_t len, int32_t* ids, int32_t cap, int32_t* n_out);
int cl_detokenize(cl_engine* e, const int32_t* ids, int32_t n, char* buf, size_t cap, size_t* len_out);

/* ---- token level (parity tests, benchmarks) --------------------------------------------- */
int cl_seq_create(cl_engine* e, cl_seq_t* out);
int cl_seq_free(cl_engine* e, cl_seq_t seq);
int cl_seq_len(cl_engine* e, cl_seq_t seq, int32_t* len_out);
/* Append n prompt tokens to the sequence.  logits_out (host, may be NULL) receives the
 * vocab_size fp32 logits of the LAST position. */
int cl_prefill(cl_engine* e, cl_seq_t seq, const int32_t* ids, int32_t n, float* logits_out);
/* The prompts of n_seqs sequences in ONE pass of the tensor-core path (the scheduler's admission of a burst of short
 * chats): ids = the prompts back to back, lens[i] tokens for seqs[i]; at most 4096 rows in total and n_seqs <= max_batch.
 * logits_out (host, may be NULL): [n_seqs][vocab_size] logits of every prompt's last position.  Results are
 * bit-identical to cl_prefill on each prompt alone through the same (tile) path. */
int cl_prefill_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs, const int32_t* ids, const int32_t* lens, float* logits_out);
/* Append one token and compute the next-token logits (host, may be NULL);
 * argmax_out (may be NULL) receives the greedy next id (lowest index on ties). */
int cl_decode_step(cl_engine* e, cl_seq_t seq, int32_t id, float* logits_out, int32_t* argmax_out);
/* Run n_steps greedy decode steps entirely on the device (each step feeds its argmax to the
 * next); ids_out receives the n_steps generated ids.  device_ms (may be NULL) receives the
 * CUDA-event time of the loop.  This is the timed region of bench.py's `value`. */
int cl_decode_greedy(cl_engine* e, cl_seq_t seq, int32_t first_id, int32_t n_steps,
                     int32_t* ids_out, float* device_ms);
/* Batched greedy decode: n_seqs sequences advance together for n_steps (continuous-batching
 * inner loop without the scheduler).  first_ids[n_seqs]; ids_out[n_steps * n_seqs]. */
int cl_decode_greedy_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs,
                           const int32_t* first_ids, int32_t n_steps, int32_t* ids_out,
                           float* device_ms);
/* Sampled counterpart of cl_decode_greedy_batch: every step runs the batched step, then the device sampler over the
 * logits of the sequences whose s[b] is sampled (greedy entries keep the step's argmax).  ids_out[i * n_seqs + b] is
 * what cl_sample_token draws from step i's logits of seqs[b] with s[b], that sequence's whole history (prompt, earlier
 * tokens, first_ids[b] and the ids drawn before) and step = first_steps[b] + i.  A sampled entry outside the device
 * limits (CL_SAMPLE_MAX_TOP_K above) returns CL_ERR_INVALID_ARG. */
int cl_decode_sample_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs, const int32_t* first_ids,
                           const cl_sampling* s, const uint64_t* first_steps, int32_t n_steps, int32_t* ids_out,
                           float* device_ms);
/* One batched decode step with caller-chosen input tokens (teacher forcing for the parity tests of the batched
 * path): ids[n_seqs]; logits_out (host, may be NULL) receives [n_seqs][vocab_size] fp32; argmax_out (may be NULL)
 * the greedy next ids. */
int cl_decode_step_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs, const int32_t* ids, float* logits_out,
                         int32_t* argmax_out);
/* Parity aid: make the sequence hold n_tokens cached tokens whose K/V, in every layer, are the CPU oracle's
 * synthetic cache pattern (oracle/llama_oracle.c oc_seq_fake_fill: k[i] = (((i * 2654435761) >> 24 & 255) - 128) / 128,
 * v[i] = (((i * 40503) >> 8 & 255) - 128) / 128 with i = token * n_kv * head_dim + head * head_dim + dim; exact in
 * bf16).  Lets the long-context decode kernels be compared with the oracle without a long CPU prefill. */
int cl_seq_fake_fill(cl_engine* e, cl_seq_t seq, int32_t n_tokens);
/* Parity aid: cached K (which = 0) / V (which = 1) rows of `layer`, tokens t0..t0+n-1 of the sequence, gathered from
 * the paged pool: out[n][n_kv_heads*head_dim] fp32 (the bf16 cache values).  Checks EVERY position of a long prefill. */
int cl_debug_kv(cl_engine* e, cl_seq_t seq, int32_t layer, int32_t which, int32_t t0, int32_t n, float* out);
/* bench.py's roofline.dominant_kernel: n_steps greedy single-sequence steps launched eagerly with a CUDA-event pair
 * (on the launching stream) around the step's dominant kernel — decode_mega_kernel, or the per-layer kernel stack
 * on the per-op path.  kernel_ms / step_ms (may be NULL): mean per step. */
int cl_time_dominant_kernel(cl_engine* e, cl_seq_t seq, int32_t first_id, int32_t n_steps, float* kernel_ms, float* step_ms);
/* debugging / parity: copy the residual stream after `layer` (or the final norm input when
 * layer == n_layers) of the most recent single-sequence step to host (d_model floats). */
int cl_debug_hidden(cl_engine* e, float* out, int32_t n);
/* profiling aid (engine created with env CL_TIMELINE=1): %globaltimer stamps [node][4] = {CTA start,
 * dependency satisfied, inputs loaded / pages consumed, outputs written} of CTA 0 of every kernel node of
 * the most recent token step; nodes = n_layers * {qkv, attn, o, gate|up, down} + lm_head.  Returns the
 * number of int64 values written (or a negative status). */
int cl_debug_timeline(cl_engine* e, int64_t* out, int32_t n);

/* ---- single-op entry points (host buffers in/out; kernel parity tests and microbenches) --
 * Each runs exactly the CUDA kernel the token step uses.  bf16 data is passed as uint16_t.
 * `variant`: 0 = generic LDG kernel, 1 = TMA-ring streaming kernel.  iters>0 => repeat and
 * report the average device time (ms) through *ms (may be NULL). */
int cl_op_gemv(int device, int variant, const uint16_t* w, const float* x, float* y,
               int32_t n_rows, int32_t k, int32_t iters, float* ms);
/* y = resid + W x */
int cl_op_gemv_residual(int device, int variant, const uint16_t* w, const float* x,
                        const float* resid, float* y, int32_t n_rows, int32_t k);
/* xn = bf16round(rmsnorm(h) * gain); y = W xn (norm fused in the GEMV prologue) */
int cl_op_rmsnorm_gemv(int device, int variant, const uint16_t* w, const float* h,
                       const float* gain, float eps, float* y, int32_t n_rows, int32_t k);
/* w_gu interleaved rows (2i = gate_i, 2i+1 = up_i); act_i = bf16round(silu(g_i) * u_i) */
int cl_op_rmsnorm_gateup(int device, int variant, const uint16_t* w_gu, const float* h,
                         const float* gain, float eps, float* act, int32_t d_ff, int32_t k);
/* fused q|k|v projection of ONE token, exactly as the token step runs it: xn = bf16(rmsnorm(h)*gain);
 * [q|k|v] = W xn (w_qkv: logical rows q | k | v in natural dim order; the wrapper applies the engine's
 * rope-pair row interleave); RoPE at `pos`; bf16 rounding.  q_out [n_heads*head_dim] fp32 (roped),
 * k_out / v_out [n_kv*head_dim] bf16 as appended to the paged cache. */
int cl_op_qkv_rope_append(int device, int variant, const uint16_t* w_qkv, const float* h, const float* gain,
                          float eps, int32_t d_model, int32_t n_heads, int32_t n_kv, int32_t head_dim,
                          int32_t pos, float rope_theta, float* q_out, uint16_t* k_out, uint16_t* v_out);
/* paged GQA decode attention for one sequence: q [n_heads*head_dim] fp32 (roped, bf16-rounded);
 * k_cache/v_cache [ctx_len][n_kv][head_dim] bf16 = tokens 0..ctx_len-1 (the current token included);
 * out [n_heads*head_dim] bf16-rounded fp32.  The wrapper scatters the cache into scrambled pages. */
int cl_op_attn_decode(int device, const float* q, const uint16_t* k_cache, const uint16_t* v_cache,
                      int32_t ctx_len, int32_t n_heads, int32_t n_kv, int32_t head_dim, int32_t page_size,
                      float* out);
/* prefill GEMM on tcgen05: Y[t][n] = sum_k X[t][k] W[n][k]; X,W bf16, Y fp32 */
int cl_op_gemm_bf16(int device, const uint16_t* x, const uint16_t* w, float* y, int32_t t,
                    int32_t n, int32_t k, int32_t iters, float* ms);
/* causal prefill attention: q [t][n_heads][d], k,v [t][n_kv][d] bf16 (roped), out bf16-rounded fp32 */
int cl_op_attn_prefill(int device, const uint16_t* q, const uint16_t* k, const uint16_t* v,
                       int32_t t, int32_t n_heads, int32_t n_kv, int32_t head_dim, float* out);
/* the same with the kernel chosen explicitly — variant 0: mma.sync kernel (prefill_kernels.cu, any head_dim 64|128),
 * 1: tcgen05 kernel (attn_prefill_tc.cu, head_dim 128), -1: what the engine would pick — and an optional timing loop */
int cl_op_attn_prefill_variant(int device, int variant, const uint16_t* q, const uint16_t* k, const uint16_t* v, int32_t t,
                               int32_t n_heads, int32_t n_kv, int32_t head_dim, float* out, int32_t iters, float* ms);
/* device sampler: logits [n_rows][vocab] fp32, s[n_rows], windows [n_rows][CL_SAMPLE_MAX_WINDOW] (row r's history: its
 * first n_window[r] entries), steps[n_rows] -> ids_out[r] == cl_sample_token(logits[r], vocab, &s[r], windows[r],
 * n_window[r], steps[r]).  Every row must be sampled (temperature > 0) and within the device limits, else
 * CL_ERR_INVALID_ARG.  iters > 0: also time that many launches over copies of the logits larger than L2 (*ms: mean). */
int cl_op_sample(int device, const float* logits, int32_t n_rows, int32_t vocab, const cl_sampling* s,
                 const int32_t* windows, const int32_t* n_window, const uint64_t* steps, int32_t* ids_out, int32_t iters,
                 float* ms);
/* logprobs_kernel on host logits [n_rows][vocab] fp32 with chosen[n_rows] the emitted ids: logprob[r] =
 * logits[r][chosen[r]] - logsumexp(logits[r]); top_ids / top_logprobs [n_rows][top_n] (may be NULL when top_n == 0) the
 * top_n best entries of each row, value descending, then id ascending.  top_n outside 0..CL_MAX_TOP_LOGPROBS:
 * CL_ERR_INVALID_ARG.  iters > 0: also time that many launches over copies of the logits larger than L2 (*ms: mean). */
int cl_op_logprobs(int device, const float* logits, int32_t n_rows, int32_t vocab, const int32_t* chosen, int32_t top_n,
                   float* logprob, int32_t* top_ids, float* top_logprobs, int32_t iters, float* ms);
/* synthetic weight generator (device kernel) -> host copy, for known-answer tests */
int cl_op_synth_weights(int device, uint64_t seed, int32_t tensor_key, int64_t n, float scale,
                        uint16_t* out_bf16);

/* ---- tokenizer (host logic; usable without a GPU) --------------------------------------------
 * Loader for HF `tokenizer.json` BPE tokenizers — SentencePiece-style (Llama-2 / Mistral / TinyLlama) and byte-level
 * (Llama-3) — replacing what the Ollama server does upstream of the reference's handler (api.go:108-160; SURVEY.md
 * §8f row 2).  chat_family: "llama3" | "mistral" | "zephyr" | "chatml" | NULL (auto from the added tokens). */
typedef struct cl_tokenizer cl_tokenizer;
int cl_tokenizer_load(const char* tokenizer_json_path, const char* chat_family, cl_tokenizer** out);
void cl_tokenizer_free(cl_tokenizer* t);
/* chat != 0: wrap text as one user turn + generation prompt first.  ids may be NULL to query *n_out. */
int cl_tokenizer_encode(const cl_tokenizer* t, const char* text, size_t len, int32_t add_bos, int32_t chat,
                        int32_t* ids, int32_t cap, int32_t* n_out);
/* raw surface bytes, special tokens skipped (may end inside a UTF-8 sequence); buf may be NULL to query *len_out */
int cl_tokenizer_decode(const cl_tokenizer* t, const int32_t* ids, int32_t n, char* buf, size_t cap, size_t* len_out);
int cl_tokenizer_info(const cl_tokenizer* t, int32_t* vocab_size, int32_t* bos, int32_t* eos);
/* install a tokenizer.json into an engine (replaces the byte-level fallback behind cl_generate*, cl_tokenize).
 * Call it before the engine serves requests: in-flight cl_generate calls tokenise without a lock. */
int cl_engine_load_tokenizer(cl_engine* e, const char* tokenizer_json_path, const char* chat_family);

/* ---- paged-KV allocator (host logic; usable without a GPU) ------------------------------ */
typedef struct cl_kvpool cl_kvpool;
int cl_kvpool_create(int32_t n_pages, int32_t page_size, cl_kvpool** out);
void cl_kvpool_destroy(cl_kvpool* p);
/* grow `owner`'s page list so it covers n_tokens; CL_ERR_OOM if the free list runs dry
 * (nothing is allocated in that case). */
int cl_kvpool_reserve(cl_kvpool* p, int32_t owner, int32_t n_tokens);
int cl_kvpool_release(cl_kvpool* p, int32_t owner);
int cl_kvpool_pages_of(cl_kvpool* p, int32_t owner, int32_t* pages, int32_t cap, int32_t* n_out);
int cl_kvpool_free_pages(cl_kvpool* p);
int cl_kvpool_used_pages(cl_kvpool* p);

#ifdef __cplusplus
}
#endif
#endif /* CLENGINE_H_ */
