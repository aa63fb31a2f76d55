// engine.h — internal C++ interface of libclengine.so (the C-ABI lives in include/clengine.h).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <deque>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/clengine.h"
#include "kernels.h"

namespace cl {

// Defaults of the features added in round 2.  Each has an environment switch; the default is turned on only after a GPU run
// of the parity tests and the benchmark with it (profiles/README.md records the run).
constexpr int kDefaultSchedPrefillChunk = 1024; // CL_SCHED_PREFILL_CHUNK: admission token budget per scheduler iteration (0 = whole prompts); validated r2e
constexpr int kDefaultPrefillSmallMax = 256;    // CL_PREFILL_SMALL_MAX: prompts up to this many tokens take the split-K path (0 = off); validated r2e (128 tokens: 12.1 -> 6.3 ms)
constexpr int kDefaultPrefillFused = 1;         // CL_PREFILL_FUSED bit mask: 1 = SiLU*mul (validated r2h: 63.2 -> 58.5 ms per 4096-token prefill), 2 = RoPE + cache scatter (correct but slower: r2g) fused into the prefill GEMM epilogues
constexpr int kDefaultSchedMultiPrefill = 1;    // CL_SCHED_MULTI_PREFILL: scheduler admits the prompts at the head of the queue in one tile-path pass (Engine::prefill_multi; validated r2v: 64 clients x 146-token prompts 38.5 -> 47.4 req/s)
constexpr int kDefaultSchedLingerUs = 1000;     // CL_SCHED_LINGER_US: with an empty batch, keep collecting while requests arrive within this gap (max 8x in total)
constexpr int kDefaultBatchMega = 0;            // CL_BATCH_MEGA: persistent batched decode kernel for B >= 2
constexpr int kDefaultSchedDeviceSample = 1;    // CL_SCHED_DEVICE_SAMPLE: requests within the device sampler's limits are sampled on the GPU (sample_kernels.cu); validated r3a: Ollama-default traffic at max_batch 64 21.3 -> 84.7 req/s

void set_last_error(const std::string& s);
const char* get_last_error();

#define CL_CUDA_OK(expr)                                                                          \
  do {                                                                                            \
    cudaError_t _e = (expr);                                                                      \
    if (_e != cudaSuccess) {                                                                      \
      ::cl::set_last_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                   \
      return CL_ERR_CUDA;                                                                         \
    }                                                                                             \
  } while (0)

// ---- paged-KV allocator: host-side free list + per-owner page lists (no GPU needed) -----------
class KvPool {
 public:
  KvPool(int n_pages, int page_size);
  int reserve(int owner, int n_tokens);  // CL_OK / CL_ERR_OOM (atomic: nothing taken on failure)
  int release(int owner);
  const std::vector<int>& pages_of(int owner);
  int free_pages() const { return (int)free_.size(); }
  int used_pages() const { return n_pages_ - (int)free_.size(); }
  int n_pages() const { return n_pages_; }
  int page_size() const { return page_size_; }

 private:
  int n_pages_, page_size_;
  std::vector<int> free_;  // stack; low page ids are handed out first
  std::map<int, std::vector<int>> owned_;
  std::vector<int> empty_;
};

// ---- tokenizers ---------------------------------------------------------------------------------
class Tokenizer {
 public:
  virtual ~Tokenizer() {}
  virtual std::vector<int32_t> encode(const std::string& text, bool add_bos) const = 0;
  virtual std::string decode_bytes(const std::vector<int32_t>& ids) const = 0;   // raw surface bytes (may cut a UTF-8 sequence)
  std::string decode(const std::vector<int32_t>& ids) const { return sanitize(decode_bytes(ids)); }
  static std::string sanitize(const std::string& raw);              // invalid UTF-8 / control bytes -> U+FFFD
  virtual int bos() const = 0;
  virtual int eos() const = 0;
  virtual bool is_stop(int id) const { return id == eos(); }        // Llama-3 also stops on <|eot_id|>
  // chat framing the Ollama server applies upstream of the model (role forced to "user", api.go:111-116)
  virtual std::string apply_chat_template(const std::string& user_prompt) const = 0;
  virtual int vocab_size() const = 0;
  // the surface bytes of one id on its own (log-probability entries); special tokens give their content
  virtual std::string token_bytes(int id) const { return decode_bytes({id}); }
};

// byte-level fallback (no vocab files exist offline; SURVEY.md §8f row 2): ids 0..2 = <pad>, <bos>, <eos>;
// byte b -> 3 + b.  Needs vocab >= 259.  A neutral, documented chat framing is used.
class ByteTokenizer : public Tokenizer {
 public:
  explicit ByteTokenizer(int vocab_size) : vocab_(vocab_size) {}
  std::vector<int32_t> encode(const std::string& text, bool add_bos) const override;
  std::string decode_bytes(const std::vector<int32_t>& ids) const override;
  int bos() const override { return 1; }
  int eos() const override { return 2; }
  std::string apply_chat_template(const std::string& user_prompt) const override;
  int vocab_size() const override { return vocab_; }

 private:
  int vocab_;
};

// HF tokenizer.json (BPE: SentencePiece-style and byte-level) — tokenizer.cpp.  chat_family: "llama3" | "mistral" |
// "zephyr" | "chatml" | "" (auto-detect from the added tokens).  nullptr + *err on failure.
std::unique_ptr<Tokenizer> load_hf_tokenizer(const std::string& path, const std::string& chat_family, std::string* err);

// HF config.json of a model directory -> cl_model_config (weights_io.cpp)
int model_config_from_dir(const std::string& dir, cl_model_config* out);

// ---- sampler (host; mirrors oracle oc_sample) ---------------------------------------------------
// inverse rotary frequency of dimension pair i: theta^(-2i/head_dim), with the "llama3" scaling of cl_model_config when
// rope_factor > 1 — the same expression as oracle/llama_oracle.c rope_inv_freq(), so both sides build bit-identical tables
double rope_inv_freq(const cl_model_config& c, int i);
int32_t sample_token(const float* logits, int32_t vocab, const cl_sampling& sp, const int32_t* history, int32_t n_history,
                     uint64_t step);

// ---- minimal protobuf codec for llama.v1.BaseMessage (pbmsg.cpp) -------------------------------
// GenerateOptions: the proto extension SURVEY.md §8f row 3 asks for (seed / temperature / num_predict ... are
// inexpressible on the reference's wire, api.go:193-197).  Every field has explicit presence: temperature 0
// (greedy) must be distinguishable from "not set".
struct PbGenerateOptions {
  uint32_t has = 0;   // bit i set <=> field number i present
  uint64_t seed = 0; float temperature = 0.f; int32_t top_k = 0; float top_p = 0.f; float repeat_penalty = 0.f;
  int32_t repeat_last_n = 0; int32_t num_predict = 0; bool raw = false;
  bool logprobs = false; int32_t top_logprobs = 0;   // fields 9, 10
};
struct PbGenerateRequest { std::string model, prompt; bool stream = false; PbGenerateOptions opt; };
// request options override the caller's default sampling field by field
void apply_options(const PbGenerateOptions& o, cl_sampling* sp);
struct PbTopLogprob { std::string token; float logprob = 0.f; };
struct PbTokenLogprob { std::string token; float logprob = 0.f; std::vector<PbTopLogprob> top_logprobs; };
struct PbGenerateResponse {
  std::string model, response, done_reason, worker_id;
  int64_t created_at_sec = 0; int32_t created_at_nanos = 0;
  bool done = false; int64_t total_duration = 0;
  std::vector<PbTokenLogprob> logprobs;               // field 8: one per token id the frame covers
};
bool pb_decode_request(const uint8_t* data, size_t len, PbGenerateRequest* out);  // false: not a GenerateRequest
std::vector<uint8_t> pb_encode_response(const PbGenerateResponse& r);

struct LayerWeights {
  float* attn_norm = nullptr;
  float* ffn_norm = nullptr;
  __nv_bfloat16* wqkv = nullptr;   // [(H + 2 KV) * D][d]   rows: q | k | v
  __nv_bfloat16* wo = nullptr;     // [d][H * D]
  __nv_bfloat16* wgu = nullptr;    // [2 F][d]             row 2i = gate_i, row 2i+1 = up_i
  __nv_bfloat16* wdown = nullptr;  // [d][F]
};

struct SeqState {
  bool live = false;
  int len = 0;            // tokens whose K/V are in the cache
  std::vector<int32_t> history;
};

struct Request;  // scheduler.cpp

class Engine {
 public:
  Engine() = default;
  ~Engine();
  int init(const cl_engine_config& cfg);

  // token-level API (callers hold mu_)
  int seq_create(cl_seq_t* out);
  int seq_free(cl_seq_t s);
  int seq_len(cl_seq_t s, int32_t* out) { if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ; *out = seqs_[s].len; return CL_OK; }
  int prefill(cl_seq_t s, const int32_t* ids, int n, float* logits_out);
  // several prompts in one pass of the tile path (prefill.cu); logits_out: [n_seqs][vocab] or nullptr
  int prefill_multi(int n_seqs, const cl_seq_t* ss, const int32_t* const* ids, const int* lens, float* logits_out);
  int decode_step(cl_seq_t s, int32_t id, float* logits_out, int32_t* argmax_out);
  // top_n (optional, [n_seqs], -1: not asked): logprobs_kernel after every step; lp_out[i * n_seqs + b] receives the
  // record of ids_out[i * n_seqs + b] (rows that did not ask: unspecified)
  int decode_greedy(const cl_seq_t* seqs, int n_seqs, const int32_t* first_ids, int n_steps, int32_t* ids_out,
                    float* device_ms, const int* top_n = nullptr, LogprobRecord* lp_out = nullptr);
  // sampled counterpart: step graph + device sampler per step; sps[b] greedy or within the device limits
  int decode_sample(const cl_seq_t* seqs, int n_seqs, const int32_t* first_ids, const cl_sampling* sps, const uint64_t* first_steps,
                    int n_steps, int32_t* ids_out, float* device_ms, const int* top_n = nullptr, LogprobRecord* lp_out = nullptr);
  // device sampler (sample_kernels.cu): true if the request's options fit its limits (clengine.h CL_SAMPLE_MAX_*)
  static bool sample_qualifies(const cl_sampling& sp, int vocab);
  // the sampler state of one slot (top_k 0: not sampled on the device); window = the last repeat_last_n ids of hist
  static SampleSlot sample_slot(const cl_sampling& sp, int vocab, const int32_t* hist, int n_hist, uint64_t step);
  // upload slot s's sampler state: the draw counter `step` and the penalty window = the last repeat_last_n ids of
  // hist[0, n_hist) (the history the next draw sees).  A greedy or non-qualifying sp leaves the slot off the sampler.
  int sample_setup(cl_seq_t s, const cl_sampling& sp, const int32_t* hist, int n_hist, uint64_t step);
  // draw the next token of the n slots whose last-position logits an admission has just left in d_logits_
  // (d_tok_[slot] is overwritten); ids_out (host, may be nullptr) receives them
  int sample_slots(const cl_seq_t* ss, int n, int32_t* ids_out);
  // log-probabilities (logprobs_kernel): enqueue one launch over the n slots whose logits rows a step or an admission has
  // just left in d_logits_ (the emitted id read from d_tok_[slot]) and the copy of their records to the host; after the
  // next synchronisation of the stream, lp_host(slot) holds them.  The buffers are allocated on the first call.
  int logprobs_enqueue(const cl_seq_t* ss, int n, int top_n);
  const LogprobRecord& lp_host(cl_seq_t s) const { return h_lp_rec_[s]; }
  // logprobs_enqueue, then wait for the stream: out[i] = the record of ss[i]
  int logprobs_read(const cl_seq_t* ss, int n, int top_n, LogprobRecord* out);
  int set_tensor(int layer, int kind, const uint16_t* data, int64_t n);
  int load_safetensors(const std::string& path);   // HF llama-layout checkpoint (file or directory) -> set_tensor (weights_io.cpp)
  // parity / benchmark aids (token level)
  int debug_kv(cl_seq_t s, int layer, int which, int t0, int n, float* out);   // cached K/V rows -> host [n][n_kv*head_dim]
  int seq_fake_fill(cl_seq_t s, int n_tokens);     // oracle oc_seq_fake_fill pattern into the paged cache of every layer
  int decode_step_batch(const cl_seq_t* seqs, int n_seqs, const int32_t* ids, float* logits_out, int32_t* argmax_out);
  int time_dominant_kernel(cl_seq_t s, int32_t first_id, int n_steps, float* kernel_ms, float* step_ms);
  int debug_hidden(float* out, int n);
  int debug_timeline(long long* out, int n);   // CL_TIMELINE=1: globaltimer stamps of the last step (CTA 0 of every node)
  int stats(cl_stats* out);

  // request-level (scheduler.cpp)
  // sink (optional): called on the CALLING thread with every batch of newly generated ids; nonzero return cancels
  // lp: the log-probability records of the ids (nullptr unless the request asked for them)
  struct TokenSink { int (*fn)(void* user, const int32_t* ids, const LogprobRecord* lp, int n) = nullptr; void* user = nullptr; };
  // top_n >= 0: the log-probabilities of every generated token with top_n alternatives go to lp_out (and the sink)
  int generate_ids(const int32_t* prompt, int n_prompt, const cl_sampling& sp, cl_result* out, const TokenSink* sink = nullptr,
                   int top_n = -1, cl_logprobs* lp_out = nullptr);
  void scheduler_main();
  void start_scheduler();
  void stop_scheduler();

  cl_model_config cfg{};
  std::string model_name;
  std::mutex mu_;               // serialises every GPU-touching call
  std::unique_ptr<Tokenizer> tok;
  bool device_sample_ = false;  // requests within the device sampler's limits are sampled on the GPU (CL_SCHED_DEVICE_SAMPLE)

 private:
  int alloc_weights();
  int fill_synthetic(uint64_t seed);
  int alloc_state();
  int ensure_capacity(cl_seq_t s, int n_tokens);  // reserve pages + upload block table row
  int enqueue_step(int B, bool tail);              // kernels of one token step for d_slots_[0..B)
  int enqueue_step_batched(int B);                 // B >= 2: tcgen05 projections + per-sequence glue kernels
  int run_step_graph(int B);
  bool ensure_graph(int B);
  void precapture_graphs();                       // graph launch (or eager enqueue)
  int read_logits(int slot, float* out);
  int launch_sampler(int B, const int* d_slots, bool ring);   // sampler over d_slots[0..B) (ring: write the step's ids_ring row)
  // logprobs_kernel over d_slots[0..B) (ring: write the step's record ring row, else the per-slot records)
  int launch_logprobs(int B, const int* d_slots, bool ring, int top_n);
  int ensure_logprobs();                                      // lazy allocation of the record buffers
  int decode_loop(const cl_seq_t* ss, int B, const int32_t* first_ids, int n_steps, int32_t* ids_out, float* device_ms, bool sample,
                  const int* top_n, LogprobRecord* lp_out);
  int prefill_tokenwise(cl_seq_t s, const int32_t* ids, int n, float* logits_out);
  int prefill_chunked(cl_seq_t s, const int32_t* ids, int n, float* logits_out);
  int ensure_prefill_ws(int tokens);  // tcgen05 path (prefill.cu)
  int prefill_small(cl_seq_t s, const int32_t* ids, int n, float* logits_out);    // short prompts: split-K projections (prefill.cu)
  bool prefill_path_ok() const;
  int set_single_slot(cl_seq_t s);

  int device_ = 0;
  cudaStream_t stream_ = nullptr;
  cudaEvent_t ev0_ = nullptr, ev1_ = nullptr;
  cudaEvent_t step_done_ev_ = nullptr;     // scheduler: blocking-sync event behind every batched step (scheduler.cpp)
  bool sched_blocking_sync_ = true;
  int sched_linger_us_ = 0;                // burst detection before a group admission into an empty batch (CL_SCHED_LINGER_US)
  bool sched_multi_prefill_ = false;       // group admission through prefill_multi (CL_SCHED_MULTI_PREFILL)
  int page_size_ = 32, max_batch_ = 8, max_seqs_ = 8, n_pages_ = 0, max_pages_per_seq_ = 0;
  int gemv_variant_ = 1, nsplit_ = 16;
  bool use_graph_ = true, use_pdl_ = true, skip_attn_ = false;
  int pdl_early_ = 1;
  bool use_flags_ = false, want_timeline_ = false, use_mega_ = false;
  MegaLayer* d_mega_layers_ = nullptr;
  CUtensorMap kmap_{}, vmap_{};
  bool have_kv_maps_ = false;
  long long* d_timeline_ = nullptr;
  unsigned* d_sync_ = nullptr;
  int n_sync_ = 0;
  int qkv_dim_ = 0, q_dim_ = 0, kv_dim_ = 0;

  // weights
  std::vector<void*> allocs_;
  __nv_bfloat16* embed_ = nullptr;
  __nv_bfloat16* lm_head_ = nullptr;
  float* final_norm_ = nullptr;
  std::vector<LayerWeights> layers_;
  float2* rope_ = nullptr;
  __nv_bfloat16* kpool_ = nullptr;  // [L][n_pages][KV][P][D]
  __nv_bfloat16* vpool_ = nullptr;
  size_t kv_layer_elems_ = 0;

  // per-slot state
  int* d_tok_ = nullptr; int* d_pos_ = nullptr; int* d_bt_ = nullptr; int* d_slots_ = nullptr;
  float* d_h_ = nullptr; float* d_q_ = nullptr; float* d_attn_ = nullptr; float* d_act_ = nullptr;
  float* d_logits_ = nullptr; float* d_attn_part_ = nullptr; unsigned* d_attn_cnt_ = nullptr;
  float* d_tail_val_ = nullptr; int* d_tail_idx_ = nullptr; unsigned* d_tail_cnt_ = nullptr;
  int* d_ids_ring_ = nullptr; int* d_step_counter_ = nullptr; int* d_prompt_ = nullptr;
  int ring_steps_ = 1024, prompt_cap_ = 0;
  float* h_logits_pinned_ = nullptr; int* h_ids_pinned_ = nullptr;
  // device sampler (sample_kernels.cu)
  SampleSlot* d_sample_state_ = nullptr;                 // [max_seqs]
  unsigned long long* d_sample_part_ = nullptr;          // [max_seqs][sample_nblk_][kSampleCand]
  unsigned* d_sample_cnt_ = nullptr;                     // [max_seqs]
  int* d_sample_slots_ = nullptr;                        // [max_seqs] slot list of an admission's sampler launch
  int sample_nblk_ = 0;                                  // 0: vocabulary too large for the device sampler
  // log-probabilities (logprobs_kernel), allocated by the first request that asks
  LogprobRecord* d_lp_rec_ = nullptr;                    // [max_seqs]
  LogprobRecord* d_lp_ring_ = nullptr;                   // [ring_steps][max_batch]
  LogprobRecord* h_lp_rec_ = nullptr;                    // pinned [max_seqs]
  LogprobRecord* h_lp_ring_ = nullptr;                   // pinned [ring_steps][max_batch]
  unsigned long long* d_lp_part_ = nullptr;              // [max_seqs][nblk][CL_MAX_TOP_LOGPROBS]
  float2* d_lp_stat_ = nullptr;                          // [max_seqs][nblk]
  unsigned* d_lp_cnt_ = nullptr;                         // [max_seqs]
  int* d_lp_slots_ = nullptr;                            // [max_seqs] slot list of the last logprobs_enqueue
  std::vector<int> lp_last_slots_;                       // what d_lp_slots_ holds

  // prefill workspace (allocated lazily)
  struct PrefillWs {
    int cap_tokens = 0;
    __nv_bfloat16* xn = nullptr;    // [T][d]
    float* qkv = nullptr;           // [T][qkv_dim]
    __nv_bfloat16* q = nullptr;     // [T][q_dim]
    __nv_bfloat16* attn = nullptr;  // [T][q_dim]
    float* h = nullptr;             // [T][d]
    float* gu = nullptr;            // [T][2F]
    __nv_bfloat16* act = nullptr;   // [T][F]
  };
  std::unique_ptr<PrefillWs> pws_;
  struct SmallPrefillWs { float* part = nullptr; __nv_bfloat16* xn = nullptr; __nv_bfloat16* q = nullptr; __nv_bfloat16* attn = nullptr;
                          float* h = nullptr; __nv_bfloat16* act = nullptr; int* iota = nullptr; };
  std::unique_ptr<SmallPrefillWs> sws_;
  int prefill_fused_ = 0;             // bit 0: SiLU*mul, bit 1: RoPE + cache scatter in the prefill GEMM epilogues (CL_PREFILL_FUSED)
  int prefill_small_max_ = 0;         // prompts up to this many tokens take the split-K path (CL_PREFILL_SMALL_MAX, 0 = off)
  struct BatchWs { __nv_bfloat16* xn = nullptr; __nv_bfloat16* attn = nullptr; __nv_bfloat16* act = nullptr; float* part = nullptr; float* logits = nullptr; };
  std::unique_ptr<BatchWs> bws_;
  bool use_batch_gemm_ = false;
  // persistent batched step (decode_mega_batch.cu)
  bool use_batch_mega_ = false;
  BatchMegaLayer* d_bm_layers_ = nullptr;
  CUtensorMap* d_bm_wmaps_ = nullptr;
  CUtensorMap bm_map_xn_{}, bm_map_attn_{}, bm_map_act_{};
  int enqueue_step_batch_mega(int B);
  int batch_gemm_min_ = 2;
  int prefill_chunk_tokens_ = 4096;

  std::unique_ptr<KvPool> pool_;
  std::vector<SeqState> seqs_;
  std::map<int, cudaGraphExec_t> graphs_;
  std::map<int, int> graph_nodes_;
  int prefill_min_tokens_ = 16;
  bool graph_failed_ = false;
  int last_single_slot_ = -1;
  bool slots_dirty_ = false;          // d_slots_ was rewritten outside the scheduler loop: its cached copy is stale
  cudaEvent_t* probe_ev_ = nullptr;   // time_dominant_kernel: event pair recorded around the dominant kernel of an eager step
  int probe_idx_ = 0;

  // stats
  std::atomic<int64_t> launches_{0}, tokens_generated_{0}, requests_completed_{0}, preemptions_{0};
  // scheduler accounting (cl_stats.sched_*): where the scheduler thread's time goes
  std::atomic<int64_t> sched_decode_steps_{0}, sched_decode_ns_{0}, sched_prefill_calls_{0}, sched_prefill_tokens_{0}, sched_prefill_ns_{0};
  double tok_per_sec_ewma_ = 0.0;          // measured: EWMA of decode steps/s x max_batch (diagnostic)
  double capacity_tok_per_sec_ = 0.0;      // advertised: load-independent capacity estimate (engine.cu init)
  char gpu_name_[64] = {0};
  int vram_gb_ = 0;

  // scheduler
  std::thread sched_thread_;
  std::mutex q_mu_;
  std::condition_variable q_cv_;
  std::deque<std::shared_ptr<Request>> queue_;
  std::vector<std::shared_ptr<Request>> active_;
  std::shared_ptr<Request> prefilling_;   // the one request whose prompt is being prefilled chunk by chunk (scheduler.cpp)
  int sched_prefill_chunk_ = 0;           // admission token budget per iteration while other sequences are decoding (CL_SCHED_PREFILL_CHUNK; 0 = unlimited)
  std::atomic<bool> stop_{false};
  bool sched_started_ = false;
  friend struct Request;
};

}  // namespace cl

struct cl_engine {
  cl::Engine impl;
};
struct cl_kvpool {
  cl::KvPool pool;
  std::mutex mu;
  cl_kvpool(int n, int p) : pool(n, p) {}
};
