// engine.cu — the worker-side decode engine: weights, paged KV cache, the token step (CUDA graph
// of hand-written sm_100a kernels), prefill, and the token-level entry points of the C-ABI.
//
// Replaces, behind crowdllama.UnifiedAPIHandler (/root/reference/pkg/crowdllama/api.go:19), the
// whole chain WorkerAPIHandler -> callOllamaAPI -> embedded Ollama server -> llama.cpp runner
// (api.go:45-160, /root/reference/cmd/crowdllama/main.go:283-297).
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>

#include <sys/stat.h>

#include "common.cuh"
#include "engine.h"

namespace cl {

static int pick_splits(int n_rows, int K);   // batched-decode split-K rule (defined with the batched step)

enum { K_EMBED = 0, K_LM_HEAD = 1, K_FINAL_NORM = 2, K_ATTN_NORM = 3, K_WQ = 4, K_WK = 5, K_WV = 6, K_WO = 7,
       K_FFN_NORM = 8, K_WGATE = 9, K_WUP = 10, K_WDOWN = 11 };
static constexpr float kLinearScale = 1.35e-4f;
static constexpr float kNormScale = 1.0f / 4096.0f;

static int env_int(const char* name, int dflt) {
  const char* v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

Engine::~Engine() {
  stop_scheduler();
  if (stream_) cudaStreamSynchronize(stream_);
  for (auto& kv : graphs_) cudaGraphExecDestroy(kv.second);
  if (step_done_ev_) cudaEventDestroy(step_done_ev_);
  for (void* p : allocs_) cudaFree(p);
  if (h_logits_pinned_) cudaFreeHost(h_logits_pinned_);
  if (h_ids_pinned_) cudaFreeHost(h_ids_pinned_);
  if (h_lp_rec_) cudaFreeHost(h_lp_rec_);
  if (h_lp_ring_) cudaFreeHost(h_lp_ring_);
  if (ev0_) cudaEventDestroy(ev0_);
  if (ev1_) cudaEventDestroy(ev1_);
  if (stream_) cudaStreamDestroy(stream_);
}

#define DMALLOC(ptr, bytes)                                          \
  do {                                                               \
    void* _p = nullptr;                                              \
    cudaError_t _e = cudaMalloc(&_p, (bytes));                       \
    if (_e != cudaSuccess) {                                         \
      set_last_error(std::string("cudaMalloc(") + #ptr + ", " + std::to_string((size_t)(bytes)) + "): " + cudaGetErrorString(_e)); \
      return _e == cudaErrorMemoryAllocation ? CL_ERR_OOM : CL_ERR_CUDA; \
    }                                                                \
    allocs_.push_back(_p);                                           \
    ptr = reinterpret_cast<decltype(ptr)>(_p);                       \
  } while (0)

int Engine::init(const cl_engine_config& c) {
  if (c.abi_version != CL_ABI_VERSION) { set_last_error("abi_version mismatch"); return CL_ERR_INVALID_ARG; }
  const std::string wpath = c.weights_path ? c.weights_path : "";
  struct stat wst{};
  const bool wdir = !wpath.empty() && stat(wpath.c_str(), &wst) == 0 && S_ISDIR(wst.st_mode);
  if (c.preset) {
    if (cl_model_preset(c.preset, &cfg) != CL_OK) { set_last_error("unknown preset"); return CL_ERR_UNKNOWN_MODEL; }
  } else if (c.model.n_layers == 0 && wdir) {
    // a model directory describes itself: config.json (HF LlamaConfig / MistralConfig field names)
    const int rc0 = model_config_from_dir(wpath, &cfg);
    if (rc0) return rc0;
  } else {
    cfg = c.model;
  }
  model_name = c.model_name ? c.model_name : (c.preset ? c.preset : "model");
  const int rep = cfg.n_kv_heads > 0 ? cfg.n_heads / cfg.n_kv_heads : 0;
  if (cfg.n_layers <= 0 || cfg.d_model <= 0 || cfg.n_heads <= 0 || cfg.n_kv_heads <= 0 || cfg.d_ff <= 0 ||
      cfg.vocab_size <= 1 || cfg.max_seq_len <= 0 || (cfg.head_dim != 64 && cfg.head_dim != 128) ||
      cfg.n_heads % cfg.n_kv_heads || (rep != 1 && rep != 2 && rep != 4 && rep != 8) || cfg.d_model % 16 || cfg.d_ff % 16 ||
      (cfg.vocab_size & 1)) {
    set_last_error("unsupported model shape (need head_dim 64|128, heads/kv in {1,2,4,8}, d_model,d_ff %16==0, even vocab)");
    return CL_ERR_INVALID_ARG;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) {
    cudaGetLastError();
    set_last_error("no CUDA device visible (libclengine has no CPU fallback)");
    return CL_ERR_NO_DEVICE;
  }
  device_ = c.device;
  if (device_ < 0 || device_ >= ndev) { set_last_error("bad device ordinal"); return CL_ERR_NO_DEVICE; }
  CL_CUDA_OK(cudaSetDevice(device_));
  cudaDeviceProp prop{};
  CL_CUDA_OK(cudaGetDeviceProperties(&prop, device_));
  if (prop.major != 10) {
    set_last_error(std::string("device is sm_") + std::to_string(prop.major * 10 + prop.minor) + ", kernels are built for sm_100a only");
    return CL_ERR_NO_DEVICE;
  }
  snprintf(gpu_name_, sizeof gpu_name_, "%s", prop.name);
  vram_gb_ = (int)(prop.totalGlobalMem >> 30);

  page_size_ = c.page_size ? c.page_size : 32;
  if (page_size_ != 16 && page_size_ != 32 && page_size_ != 64) { set_last_error("page_size must be 16, 32 or 64"); return CL_ERR_INVALID_ARG; }
  max_batch_ = c.max_batch > 0 ? c.max_batch : 8;
  max_seqs_ = c.max_seqs > 0 ? c.max_seqs : max_batch_;
  if (max_seqs_ < max_batch_) max_seqs_ = max_batch_;
  use_graph_ = c.use_cuda_graph >= 0 && env_int("CL_GRAPH", 1) != 0;
  use_pdl_ = env_int("CL_PDL", 1) != 0;
  pdl_early_ = env_int("CL_PDL_EARLY", 1);
  skip_attn_ = env_int("CL_SKIP_ATTN", 0) != 0;   // timing experiments only (wrong results)
  use_flags_ = env_int("CL_FLAGS", 0) != 0;      // measured slower than griddepcontrol.wait (profiles/README.md)
  want_timeline_ = env_int("CL_TIMELINE", 0) != 0;
  gemv_variant_ = c.decode_path == 1 ? 0 : 1;
  gemv_variant_ = env_int("CL_GEMV_VARIANT", gemv_variant_);
  q_dim_ = cfg.n_heads * cfg.head_dim;
  kv_dim_ = cfg.n_kv_heads * cfg.head_dim;
  qkv_dim_ = q_dim_ + 2 * kv_dim_;
  nsplit_ = std::max(1, std::min(64, sm_count() / cfg.n_kv_heads));
  nsplit_ = std::max(1, std::min(64, env_int("CL_ATTN_NSPLIT", nsplit_)));
  // decided AFTER nsplit_ is final: the persistent kernel's lane-parallel combine and part buffer are sized by it
  use_mega_ = env_int("CL_MEGA", 1) != 0 &&
              mega_supported(cfg.d_model, cfg.d_ff, cfg.head_dim, cfg.n_heads, cfg.n_kv_heads, page_size_, nsplit_);
  max_pages_per_seq_ = (cfg.max_seq_len + page_size_ - 1) / page_size_;

  const size_t kv_bytes_per_token = (size_t)2 * cfg.n_layers * kv_dim_ * 2;
  int64_t pool_bytes = c.kv_pool_bytes;
  if (pool_bytes <= 0) pool_bytes = (int64_t)max_seqs_ * max_pages_per_seq_ * page_size_ * (int64_t)kv_bytes_per_token;
  n_pages_ = (int)(pool_bytes / ((int64_t)page_size_ * (int64_t)kv_bytes_per_token));
  if (n_pages_ < 1) { set_last_error("kv_pool_bytes too small for one page"); return CL_ERR_INVALID_ARG; }

  CL_CUDA_OK(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking));
  CL_CUDA_OK(cudaEventCreate(&ev0_));
  CL_CUDA_OK(cudaEventCreate(&ev1_));
  int rc = alloc_weights();
  if (rc) return rc;
  // weights_path: HF llama-layout safetensors (file or model directory, weights_io.cpp); else seeded synthetic weights
  rc = wpath.empty() ? fill_synthetic(c.weights_seed) : load_safetensors(wpath);
  if (rc) return rc;
  rc = alloc_state();
  if (rc) return rc;
  if (cfg.head_dim == 128 && page_size_ == 32) {   // pool-wide KV tensor maps: persistent kernel + tensor-core batched attention
    const uint64_t rows = (uint64_t)cfg.n_layers * n_pages_ * cfg.n_kv_heads * page_size_;
    have_kv_maps_ = rows < (1ull << 31) && make_tmap_2d_bf16(&kmap_, kpool_, rows, cfg.head_dim, 64, 32) &&
                    make_tmap_2d_bf16(&vmap_, vpool_, rows, cfg.head_dim, 64, 32);
  }
  if (use_mega_ && !have_kv_maps_) {
    fprintf(stderr, "[clengine] KV tensor maps unavailable: using the per-op decode path\n");
    use_mega_ = false;
  }
  if (use_mega_ && !mega_prepare_device()) {
    fprintf(stderr, "[clengine] persistent decode kernel does not fit one CTA per SM on this device: using the per-op decode path\n");
    use_mega_ = false;
  }
  if (use_mega_) {
    std::vector<MegaLayer> ml(cfg.n_layers);
    for (int l = 0; l < cfg.n_layers; ++l)
      ml[l] = MegaLayer{layers_[l].wqkv, layers_[l].wo, layers_[l].wgu, layers_[l].wdown, layers_[l].attn_norm, layers_[l].ffn_norm,
                        kpool_ + (size_t)l * kv_layer_elems_, vpool_ + (size_t)l * kv_layer_elems_};
    DMALLOC(d_mega_layers_, ml.size() * sizeof(MegaLayer));
    CL_CUDA_OK(cudaMemcpy(d_mega_layers_, ml.data(), ml.size() * sizeof(MegaLayer), cudaMemcpyHostToDevice));
  }
  pool_.reset(new KvPool(n_pages_, page_size_));
  seqs_.assign(max_seqs_, SeqState());
  tok.reset(new ByteTokenizer(cfg.vocab_size));
  if (wdir) {   // a model directory brings its vocabulary: tokenizer.json replaces the byte-level fallback
    const std::string tj = wpath + "/tokenizer.json";
    if (stat(tj.c_str(), &wst) == 0) {
      std::string err;
      std::unique_ptr<Tokenizer> t = load_hf_tokenizer(tj, "", &err);
      if (!t) { set_last_error("tokenizer.json: " + err); return CL_ERR_IO; }
      if (t->vocab_size() > cfg.vocab_size) { set_last_error("tokenizer.json has more ids than the model's vocabulary"); return CL_ERR_IO; }
      tok = std::move(t);
    }
  }
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  {
    // Advertised throughput = CAPACITY, and load-INDEPENDENT: what this worker can deliver with a full batch, estimated
    // from the device's memory bandwidth and the model's bytes per token (70 % of the HBM roofline of one decode step x
    // max_batch).  Round 1 advertised the measured decode steps/s x max_batch; a step at B = 32 takes 1.6x as long as at
    // B = 1, so busy workers advertised LESS than idle ones, crossed a half-octave bucket, and FindBestWorker's strict
    // maximum (manager.go:369-377) sent every request of a refresh interval to one idle worker (8 peers, r2k: 96 of 192
    // requests on one worker).  Identical GPUs now advertise identical numbers and tie, which is what the reference's
    // constants (peer.go:319-343) did; the measured rate stays available as cl_stats.measured_tokens_per_sec.
    const double params = (double)cfg.n_layers * ((double)qkv_dim_ * cfg.d_model + (double)cfg.d_model * q_dim_ + 3.0 * cfg.d_ff * cfg.d_model) +
                          (double)cfg.vocab_size * cfg.d_model;
    double bw = 2.0 * (double)prop.memoryClockRate * 1e3 * (double)prop.memoryBusWidth / 8.0;   // bytes/s (DDR)
    if (!(bw > 1e11)) bw = 6.5e12;
    capacity_tok_per_sec_ = 0.7 * bw / (2.0 * params) * (double)max_batch_;
    tok_per_sec_ewma_ = 0.0;
  }
  // defaults of the round-2 features: see kDefault* in engine.h (flipped on once a GPU run has validated them)
  sched_prefill_chunk_ = env_int("CL_SCHED_PREFILL_CHUNK", kDefaultSchedPrefillChunk);
  device_sample_ = env_int("CL_SCHED_DEVICE_SAMPLE", kDefaultSchedDeviceSample) != 0 && sample_nblk_ > 0;
  if (sched_prefill_chunk_ > 0 && sched_prefill_chunk_ < 16) sched_prefill_chunk_ = 16;
  prefill_small_max_ = std::min(256, env_int("CL_PREFILL_SMALL_MAX", kDefaultPrefillSmallMax));
  prefill_fused_ = env_int("CL_PREFILL_FUSED", kDefaultPrefillFused);
  if (c.start_scheduler) start_scheduler();
  return CL_OK;
}

int Engine::alloc_weights() {
  const size_t d = cfg.d_model, F = cfg.d_ff, V = cfg.vocab_size;
  DMALLOC(embed_, V * d * 2);
  DMALLOC(lm_head_, V * d * 2);
  DMALLOC(final_norm_, d * 4);
  layers_.resize(cfg.n_layers);
  for (auto& L : layers_) {
    DMALLOC(L.attn_norm, d * 4);
    DMALLOC(L.ffn_norm, d * 4);
    DMALLOC(L.wqkv, (size_t)qkv_dim_ * d * 2);
    DMALLOC(L.wo, d * (size_t)q_dim_ * 2);
    DMALLOC(L.wgu, 2 * F * d * 2);
    DMALLOC(L.wdown, d * F * 2);
  }
  // RoPE table: computed on the host in double, rounded to fp32 — the same expression as
  // oracle/llama_oracle.c build_rope(), so both sides use bit-identical cos/sin.
  const int half = cfg.head_dim / 2;
  std::vector<float2> tab((size_t)cfg.max_seq_len * half);
  for (int p = 0; p < cfg.max_seq_len; ++p)
    for (int i = 0; i < half; ++i) {
      const double ang = (double)p * rope_inv_freq(cfg, i);
      tab[(size_t)p * half + i] = make_float2((float)cos(ang), (float)sin(ang));
    }
  DMALLOC(rope_, tab.size() * sizeof(float2));
  CL_CUDA_OK(cudaMemcpy(rope_, tab.data(), tab.size() * sizeof(float2), cudaMemcpyHostToDevice));
  kv_layer_elems_ = (size_t)n_pages_ * cfg.n_kv_heads * page_size_ * cfg.head_dim;
  DMALLOC(kpool_, kv_layer_elems_ * cfg.n_layers * 2);
  DMALLOC(vpool_, kv_layer_elems_ * cfg.n_layers * 2);
  CL_CUDA_OK(cudaMemsetAsync(kpool_, 0, kv_layer_elems_ * cfg.n_layers * 2, stream_));
  CL_CUDA_OK(cudaMemsetAsync(vpool_, 0, kv_layer_elems_ * cfg.n_layers * 2, stream_));
  return CL_OK;
}

int Engine::fill_synthetic(uint64_t seed) {
  const int d = cfg.d_model, F = cfg.d_ff, V = cfg.vocab_size;
  int n = 0;
  n += launch_synth_bf16(embed_, (int64_t)V * d, d, 1, 0, seed, K_EMBED, kLinearScale, stream_);
  n += launch_synth_bf16(lm_head_, (int64_t)V * d, d, 1, 0, seed, K_LM_HEAD, kLinearScale, stream_);
  n += launch_synth_gain(final_norm_, d, seed, K_FINAL_NORM, kNormScale, stream_);
  for (int l = 0; l < cfg.n_layers; ++l) {
    auto& L = layers_[l];
    const int b = l * 16;
    n += launch_synth_gain(L.attn_norm, d, seed, b + K_ATTN_NORM, kNormScale, stream_);
    n += launch_synth_gain(L.ffn_norm, d, seed, b + K_FFN_NORM, kNormScale, stream_);
    // q|k|v rows are stored rope-pair-interleaved per head (kernels.h: QkvEpi)
    n += launch_synth_bf16(L.wqkv, (int64_t)q_dim_ * d, d, 1, 0, seed, b + K_WQ, kLinearScale, stream_, cfg.head_dim);
    n += launch_synth_bf16(L.wqkv + (size_t)q_dim_ * d, (int64_t)kv_dim_ * d, d, 1, 0, seed, b + K_WK, kLinearScale, stream_, cfg.head_dim);
    n += launch_synth_bf16(L.wqkv + (size_t)(q_dim_ + kv_dim_) * d, (int64_t)kv_dim_ * d, d, 1, 0, seed, b + K_WV, kLinearScale, stream_, cfg.head_dim);
    n += launch_synth_bf16(L.wo, (int64_t)d * q_dim_, q_dim_, 1, 0, seed, b + K_WO, kLinearScale, stream_);
    n += launch_synth_bf16(L.wgu, (int64_t)F * d, d, 2, 0, seed, b + K_WGATE, kLinearScale, stream_);
    n += launch_synth_bf16(L.wgu, (int64_t)F * d, d, 2, 1, seed, b + K_WUP, kLinearScale, stream_);
    n += launch_synth_bf16(L.wdown, (int64_t)d * F, F, 1, 0, seed, b + K_WDOWN, kLinearScale, stream_);
  }
  launches_ += n;
  CL_CUDA_OK(cudaGetLastError());
  return CL_OK;
}

int Engine::set_tensor(int layer, int kind, const uint16_t* data, int64_t n) {
  const int64_t d = cfg.d_model, F = cfg.d_ff, V = cfg.vocab_size;
  auto copy16 = [&](__nv_bfloat16* dst, int64_t want) -> int {
    if (n != want) { set_last_error("set_tensor: wrong element count"); return CL_ERR_INVALID_ARG; }
    CL_CUDA_OK(cudaMemcpy(dst, data, (size_t)n * 2, cudaMemcpyHostToDevice));
    return CL_OK;
  };
  auto copy_gain = [&](float* dst, int64_t want) -> int {
    if (n != want) { set_last_error("set_tensor: wrong element count"); return CL_ERR_INVALID_ARG; }
    std::vector<float> f((size_t)n);
    for (int64_t i = 0; i < n; ++i) { uint32_t u = (uint32_t)data[i] << 16; memcpy(&f[i], &u, 4); }
    CL_CUDA_OK(cudaMemcpy(dst, f.data(), (size_t)n * 4, cudaMemcpyHostToDevice));
    return CL_OK;
  };
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  if (kind == K_EMBED) return copy16(embed_, V * d);
  if (kind == K_LM_HEAD) return copy16(lm_head_, V * d);
  if (kind == K_FINAL_NORM) return copy_gain(final_norm_, d);
  if (layer < 0 || layer >= cfg.n_layers) { set_last_error("set_tensor: bad layer"); return CL_ERR_INVALID_ARG; }
  auto& L = layers_[layer];
  switch (kind) {
    case K_ATTN_NORM: return copy_gain(L.attn_norm, d);
    case K_FFN_NORM: return copy_gain(L.ffn_norm, d);
    case K_WQ:
    case K_WK:
    case K_WV: {
      const int64_t rows = kind == K_WQ ? q_dim_ : kv_dim_;
      if (n != rows * d) { set_last_error("set_tensor: wrong element count"); return CL_ERR_INVALID_ARG; }
      __nv_bfloat16* dst = L.wqkv + (kind == K_WQ ? 0 : kind == K_WK ? (size_t)q_dim_ * d : (size_t)(q_dim_ + kv_dim_) * d);
      // rope-pair interleave per head: logical row (head, w) -> head*hd + (w < hd/2 ? 2w : 2(w - hd/2) + 1)
      std::vector<uint16_t> perm((size_t)n);
      const int hd = cfg.head_dim, half = hd / 2;
      for (int64_t r = 0; r < rows; ++r) {
        const int64_t head = r / hd;
        const int w = (int)(r % hd);
        const int64_t rr = head * hd + (w < half ? 2 * w : 2 * (w - half) + 1);
        memcpy(&perm[(size_t)rr * d], data + (size_t)r * d, (size_t)d * 2);
      }
      CL_CUDA_OK(cudaMemcpy(dst, perm.data(), (size_t)n * 2, cudaMemcpyHostToDevice));
      return CL_OK;
    }
    case K_WO: return copy16(L.wo, d * q_dim_);
    case K_WDOWN: return copy16(L.wdown, d * F);
    case K_WGATE:
    case K_WUP: {
      if (n != F * d) { set_last_error("set_tensor: wrong element count"); return CL_ERR_INVALID_ARG; }
      // interleave on the device side with a strided 2-D copy: row r -> row 2r (+1 for up)
      CL_CUDA_OK(cudaMemcpy2D(L.wgu + (kind == K_WUP ? d : 0), (size_t)2 * d * 2, data, (size_t)d * 2, (size_t)d * 2, (size_t)F,
                              cudaMemcpyHostToDevice));
      return CL_OK;
    }
    default: set_last_error("set_tensor: bad kind"); return CL_ERR_INVALID_ARG;
  }
}

int Engine::alloc_state() {
  const size_t S = max_seqs_, d = cfg.d_model;
  DMALLOC(d_tok_, S * 4);
  DMALLOC(d_pos_, S * 4);
  DMALLOC(d_bt_, S * max_pages_per_seq_ * 4);
  DMALLOC(d_slots_, (size_t)max_batch_ * 4);
  DMALLOC(d_h_, S * d * 4);
  DMALLOC(d_q_, S * q_dim_ * 4);
  DMALLOC(d_attn_, S * q_dim_ * 4);
  DMALLOC(d_act_, S * (size_t)cfg.d_ff * 4);
  DMALLOC(d_logits_, S * (size_t)cfg.vocab_size * 4);
  const int rep = cfg.n_heads / cfg.n_kv_heads;
  DMALLOC(d_attn_part_, S * cfg.n_kv_heads * nsplit_ * rep * (cfg.head_dim + 2) * 4);
  DMALLOC(d_attn_cnt_, S * cfg.n_kv_heads * 4);
  DMALLOC(d_tail_val_, S * 64 * 4);
  DMALLOC(d_tail_idx_, S * 64 * 4);
  DMALLOC(d_tail_cnt_, S * 4);
  DMALLOC(d_ids_ring_, (size_t)ring_steps_ * max_batch_ * 4);
  DMALLOC(d_step_counter_, 4);
  n_sync_ = std::max(cfg.n_layers * 5 + 1 + cfg.n_layers * max_batch_, cfg.n_layers * 10 + 4);   // megakernel: 6 barriers + 4 tile counters per layer + lookahead frontier
  DMALLOC(d_sync_, (size_t)n_sync_ * 4);
  CL_CUDA_OK(cudaMemsetAsync(d_sync_, 0, (size_t)n_sync_ * 4, stream_));
  if (want_timeline_) {
    DMALLOC(d_timeline_, (size_t)(cfg.n_layers * 5 + 1) * 4 * 8);   // >= n_layers * 16 stamps for the megakernel view
    CL_CUDA_OK(cudaMemsetAsync(d_timeline_, 0, (size_t)(cfg.n_layers * 5 + 1) * 4 * 8, stream_));
  }
  batch_gemm_min_ = env_int("CL_BATCH_GEMM_MIN", 2);
  // token tile of the projections = 32 / 64 / 128 rows (gemm_tcgen05.cu picks it from the step's batch size)
  use_batch_gemm_ = env_int("CL_BATCH_GEMM", 1) != 0 && max_batch_ >= 2 && gemm_tcgen05_supported(max_batch_, cfg.d_model, cfg.d_model) &&
                    max_batch_ <= 128;
  if (use_batch_gemm_) {
    bws_.reset(new BatchWs());
    const size_t Bm = std::max(max_batch_, 32), widest = std::max<size_t>((size_t)qkv_dim_, std::max<size_t>(2 * (size_t)cfg.d_ff, d));   // 32 rows: the persistent batched kernel's token tile
    DMALLOC(bws_->xn, Bm * d * 2);
    DMALLOC(bws_->attn, Bm * q_dim_ * 2);
    DMALLOC(bws_->act, Bm * (size_t)cfg.d_ff * 2);
    CL_CUDA_OK(cudaMemsetAsync(bws_->xn, 0, Bm * d * 2, stream_));
    CL_CUDA_OK(cudaMemsetAsync(bws_->attn, 0, Bm * q_dim_ * 2, stream_));
    CL_CUDA_OK(cudaMemsetAsync(bws_->act, 0, Bm * (size_t)cfg.d_ff * 2, stream_));
    // split-K partial workspace of the four projections (pick_splits)
    size_t part_floats = 4 * Bm * widest;
    for (int nk : {0, 1, 2, 3}) {
      const int N = nk == 0 ? qkv_dim_ : nk == 2 ? 2 * cfg.d_ff : d, K = nk == 1 ? q_dim_ : nk == 3 ? cfg.d_ff : d;
      part_floats = std::max(part_floats, (size_t)pick_splits(N, K) * Bm * (size_t)N);
    }
    DMALLOC(bws_->part, part_floats * 4);
    DMALLOC(bws_->logits, Bm * (size_t)cfg.vocab_size * 4);
    // persistent batched step: tensor maps of every weight matrix (device array) and of the three token operands
    use_batch_mega_ = env_int("CL_BATCH_MEGA", kDefaultBatchMega) != 0 && cfg.head_dim == 128 && page_size_ == 32 && max_batch_ <= 32 &&
                      batch_mega_supported(cfg.d_model, cfg.d_ff, cfg.head_dim, cfg.n_heads, cfg.n_kv_heads, page_size_, cfg.vocab_size);
    if (use_batch_mega_) {
      auto kbp = [&](int N, int K) { const int nkb = K / 64, sp = pick_splits(N, K); return (nkb + sp - 1) / sp; };
      if (kbp(qkv_dim_, cfg.d_model) > 25 || kbp(cfg.d_model, q_dim_) > 25 || kbp(2 * cfg.d_ff, cfg.d_model) > 25 || kbp(cfg.d_model, cfg.d_ff) > 25)
        use_batch_mega_ = false;   // a split's token operand must fit the kernel's 25 resident tiles
    }
    if (use_batch_mega_) {
      std::vector<CUtensorMap> wm((size_t)cfg.n_layers * 4 + 1);
      std::vector<BatchMegaLayer> bl(cfg.n_layers);
      bool ok = batch_mega_prepare_device();
      for (int l = 0; l < cfg.n_layers && ok; ++l) {
        const auto& L = layers_[l];
        ok = make_wmap(&wm[(size_t)l * 4 + 0], L.wqkv, qkv_dim_, cfg.d_model) && make_wmap(&wm[(size_t)l * 4 + 1], L.wo, cfg.d_model, q_dim_) &&
             make_wmap(&wm[(size_t)l * 4 + 2], L.wgu, 2 * cfg.d_ff, cfg.d_model) && make_wmap(&wm[(size_t)l * 4 + 3], L.wdown, cfg.d_model, cfg.d_ff);
        bl[l] = BatchMegaLayer{L.attn_norm, L.ffn_norm, kpool_ + (size_t)l * kv_layer_elems_, vpool_ + (size_t)l * kv_layer_elems_};
      }
      ok = ok && make_wmap(&wm[(size_t)cfg.n_layers * 4], lm_head_, cfg.vocab_size, cfg.d_model) &&
           make_tmap_2d_bf16(&bm_map_xn_, bws_->xn, 32, cfg.d_model, 64, 32) && make_tmap_2d_bf16(&bm_map_attn_, bws_->attn, 32, q_dim_, 64, 32) &&
           make_tmap_2d_bf16(&bm_map_act_, bws_->act, 32, cfg.d_ff, 64, 32);
      if (ok) {
        DMALLOC(d_bm_wmaps_, wm.size() * sizeof(CUtensorMap));
        DMALLOC(d_bm_layers_, bl.size() * sizeof(BatchMegaLayer));
        CL_CUDA_OK(cudaMemcpy(d_bm_wmaps_, wm.data(), wm.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice));
        CL_CUDA_OK(cudaMemcpy(d_bm_layers_, bl.data(), bl.size() * sizeof(BatchMegaLayer), cudaMemcpyHostToDevice));
      } else {
        fprintf(stderr, "[clengine] persistent batched decode kernel unavailable on this device / shape: using the per-kernel batched step\n");
        use_batch_mega_ = false;
      }
    }
  }
  prompt_cap_ = cfg.max_seq_len;
  DMALLOC(d_prompt_, (size_t)prompt_cap_ * 4);
  CL_CUDA_OK(cudaMemsetAsync(d_tok_, 0, S * 4, stream_));
  CL_CUDA_OK(cudaMemsetAsync(d_pos_, 0, S * 4, stream_));
  CL_CUDA_OK(cudaMemsetAsync(d_bt_, 0, S * max_pages_per_seq_ * 4, stream_));
  CL_CUDA_OK(cudaMemsetAsync(d_slots_, 0, (size_t)max_batch_ * 4, stream_));
  CL_CUDA_OK(cudaMemsetAsync(d_attn_cnt_, 0, S * cfg.n_kv_heads * 4, stream_));
  CL_CUDA_OK(cudaMemsetAsync(d_tail_cnt_, 0, S * 4, stream_));
  CL_CUDA_OK(cudaMemsetAsync(d_step_counter_, 0, 4, stream_));
  CL_CUDA_OK(cudaMallocHost(&h_logits_pinned_, (size_t)cfg.vocab_size * 4));
  CL_CUDA_OK(cudaMallocHost(&h_ids_pinned_, (size_t)ring_steps_ * max_batch_ * 4));
  sample_nblk_ = sample_blocks(cfg.vocab_size);
  if (sample_nblk_ > 0) {
    DMALLOC(d_sample_state_, S * sizeof(SampleSlot));
    DMALLOC(d_sample_part_, S * sample_nblk_ * kSampleCand * sizeof(unsigned long long));
    DMALLOC(d_sample_cnt_, S * 4);
    DMALLOC(d_sample_slots_, S * 4);
    CL_CUDA_OK(cudaMemsetAsync(d_sample_state_, 0, S * sizeof(SampleSlot), stream_));
    CL_CUDA_OK(cudaMemsetAsync(d_sample_cnt_, 0, S * 4, stream_));
  }
  return CL_OK;
}

// ---- sequences ----------------------------------------------------------------------------------
int Engine::seq_create(cl_seq_t* out) {
  for (int i = 0; i < max_seqs_; ++i)
    if (!seqs_[i].live) {
      if (d_sample_state_) CL_CUDA_OK(cudaMemsetAsync(d_sample_state_ + i, 0, sizeof(SampleSlot), stream_));   // off the device sampler
      seqs_[i] = SeqState();
      seqs_[i].live = true;
      *out = i;
      return CL_OK;
    }
  set_last_error("no free sequence slot (max_seqs)");
  return CL_ERR_OOM;
}
int Engine::seq_free(cl_seq_t s) {
  if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
  pool_->release(s);
  seqs_[s] = SeqState();
  return CL_OK;
}

int Engine::ensure_capacity(cl_seq_t s, int n_tokens) {
  if (n_tokens > cfg.max_seq_len) { set_last_error("sequence exceeds max_seq_len"); return CL_ERR_TOO_LONG; }
  const size_t before = pool_->pages_of(s).size();
  const int rc = pool_->reserve(s, n_tokens);
  if (rc) { set_last_error("KV page pool exhausted"); return rc; }
  const auto& pages = pool_->pages_of(s);
  if (pages.size() != before)
    CL_CUDA_OK(cudaMemcpyAsync(d_bt_ + (size_t)s * max_pages_per_seq_ + before, pages.data() + before,
                               (pages.size() - before) * 4, cudaMemcpyHostToDevice, stream_));
  return CL_OK;
}

// ---- one token step for the sequences listed in d_slots_[0..B) -----------------------------------
int Engine::enqueue_step(int B, bool tail) {
  if (B >= 2 && tail && use_batch_mega_ && have_kv_maps_ && bws_) return enqueue_step_batch_mega(B);
  if (B >= batch_gemm_min_ && tail && use_batch_gemm_ && bws_) return enqueue_step_batched(B);   // from B = 2: 3.58 vs 3.94 ms at ctx 256, 3.72 vs 4.29 at ctx 4096 against two GEMV passes (r2p)
  const int d = cfg.d_model, F = cfg.d_ff, L_ = cfg.n_layers;
  int n = 0, r;
#define CL_LAUNCH(call) do { r = (call); if (r < 0) { set_last_error(std::string(#call) + ": " + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; } n += r; } while (0)
  // StepSync: counter-based dependencies inside the step (kernels.h).  Only with PDL (the consumers must
  // already be resident to profit) and never for the first kernel after embed / the tail (stream order).
  const bool flags = use_flags_ && use_pdl_;
  const bool defer_combine = flags && gemv_variant_ == 1 && gemv_variant_supported(1, d, q_dim_) && nsplit_ <= 32 &&
                             (q_dim_ + sm_count() - 1) / sm_count() <= 64;
  auto cnt = [&](int l, int k) -> unsigned* { return flags ? d_sync_ + (size_t)l * 5 + k : nullptr; };
  auto tl = [&](int l, int k) -> long long* { return d_timeline_ ? d_timeline_ + ((size_t)l * 5 + k) * 4 : nullptr; };
  const unsigned* prev_cnt = nullptr;
  int prev_n = 0, nc = 0;
  CL_LAUNCH(launch_embed(embed_, d, d_tok_, d_h_, d, d_slots_, B, stream_));
  const bool mega = use_mega_ && B == 1 && !skip_attn_ && d_mega_layers_ != nullptr;
  if (probe_ev_) cudaEventRecord(probe_ev_[probe_idx_], stream_);
  if (mega) {
    MegaArgs m;
    m.layers = d_mega_layers_; m.n_layers = L_; m.q_dim = q_dim_; m.qkv_dim = qkv_dim_; m.n_heads = cfg.n_heads; m.n_kv = cfg.n_kv_heads;
    m.nsplit = nsplit_; m.eps = cfg.rms_eps; m.rope = rope_; m.pos = d_pos_; m.block_tables = d_bt_; m.bt_stride = max_pages_per_seq_;
    m.slots = d_slots_; m.h = d_h_; m.q = d_q_; m.attn_x = d_attn_; m.act = d_act_; m.part = d_attn_part_; m.bars = d_sync_; m.tile_ctr = d_sync_ + (size_t)L_ * 6; m.pf_ctr = d_sync_ + (size_t)L_ * 10; m.max_flight = env_int("CL_MEGA_MAX_FLIGHT", 2); m.pause_in_barrier = env_int("CL_MEGA_PAUSE", 1); m.pf_min = env_int("CL_MEGA_PF_MIN", 900); m.pf_budget = env_int("CL_MEGA_PF_BUDGET", 4096);
    m.tl = d_timeline_; m.tl_cta = env_int("CL_TIMELINE_CTA", 0);
    m.kv_layer_rows = (long long)n_pages_ * cfg.n_kv_heads * page_size_; m.kmap = kmap_; m.vmap = vmap_;
    CL_LAUNCH(launch_decode_mega(m, stream_));
  }
  for (int l = 0; l < (mega ? 0 : L_); ++l) {
    const auto& L = layers_[l];
    GemvArgs g;
    g.slots = d_slots_; g.batch = B; g.pdl_early = pdl_early_;
    // (1) RMSNorm + fused q|k|v projection; epilogue: RoPE + bf16 round + q out + KV append into the paged cache
    g.W = L.wqkv; g.N = qkv_dim_; g.K = d; g.h = d_h_; g.gain = L.attn_norm; g.eps = cfg.rms_eps;
    g.y = d_q_; g.x_stride = d; g.y_stride = q_dim_;
    g.qkv.rope = rope_; g.qkv.pos = d_pos_; g.qkv.block_tables = d_bt_; g.qkv.bt_stride = max_pages_per_seq_;
    g.qkv.kpool = kpool_ + (size_t)l * kv_layer_elems_; g.qkv.vpool = vpool_ + (size_t)l * kv_layer_elems_;
    g.qkv.n_heads = cfg.n_heads; g.qkv.n_kv = cfg.n_kv_heads; g.qkv.head_dim = cfg.head_dim; g.qkv.page_size = page_size_;
    g.sync.wait = prev_cnt; g.sync.n_wait = (unsigned)prev_n; g.sync.signal = cnt(l, 0); g.tl = tl(l, 0);
    CL_LAUNCH(launch_gemv(gemv_variant_, EPI_QKV, true, g, stream_, use_pdl_, &nc));
    prev_cnt = cnt(l, 0); prev_n = nc;
    // (2) paged GQA attention over tokens 0..pos
    AttnDecodeArgs a;
    a.q = d_q_; a.q_stride = q_dim_;
    a.kpool = kpool_ + (size_t)l * kv_layer_elems_; a.vpool = vpool_ + (size_t)l * kv_layer_elems_;
    a.block_tables = d_bt_; a.bt_stride = max_pages_per_seq_; a.pos = d_pos_;
    a.out = d_attn_; a.out_stride = q_dim_; a.part = d_attn_part_; a.counters = d_attn_cnt_;
    a.slots = d_slots_; a.batch = B; a.n_heads = cfg.n_heads; a.n_kv = cfg.n_kv_heads; a.head_dim = cfg.head_dim;
    a.page_size = page_size_; a.nsplit = nsplit_; a.pdl_early = pdl_early_;
    a.sync.wait = prev_cnt; a.sync.n_wait = (unsigned)prev_n;
    a.sync.signal = defer_combine ? cnt(l, 1) : nullptr; a.tl = tl(l, 1);
    if (!skip_attn_) CL_LAUNCH(launch_attn_decode(a, stream_, use_pdl_));
    // (3) o projection + residual (prologue: cross-split combine of the attention partials when deferred)
    GemvArgs o;
    o.slots = d_slots_; o.batch = B; o.pdl_early = pdl_early_;
    o.W = L.wo; o.N = d; o.K = q_dim_; o.x = d_attn_; o.x_stride = q_dim_; o.y = d_h_; o.resid = d_h_; o.y_stride = d;
    if (defer_combine && !skip_attn_) {
      o.sync.wait = cnt(l, 1); o.sync.n_wait = (unsigned)(cfg.n_kv_heads * nsplit_ * B);
      o.comb.part = d_attn_part_; o.comb.nsplit = nsplit_; o.comb.n_kv = cfg.n_kv_heads; o.comb.rep = cfg.n_heads / cfg.n_kv_heads;
      o.comb.head_dim = cfg.head_dim; o.comb.x_out = d_attn_; o.comb.phase = d_sync_ + (size_t)L_ * 5 + 1 + (size_t)l * max_batch_;
    } else {
      // the attention kernel combined in-kernel and publishes nothing: fall back to grid completion
      o.sync.wait = nullptr;
    }
    o.sync.signal = cnt(l, 2); o.tl = tl(l, 2);
    CL_LAUNCH(launch_gemv(gemv_variant_, EPI_RESID, false, o, stream_, use_pdl_, &nc));
    prev_cnt = cnt(l, 2); prev_n = nc;
    // (4) RMSNorm + gate/up + SiLU*mul
    GemvArgs u;
    u.slots = d_slots_; u.batch = B; u.pdl_early = pdl_early_;
    u.W = L.wgu; u.N = 2 * F; u.K = d; u.h = d_h_; u.gain = L.ffn_norm; u.eps = cfg.rms_eps; u.y = d_act_;
    u.x_stride = d; u.y_stride = F;
    u.sync.wait = prev_cnt; u.sync.n_wait = (unsigned)prev_n; u.sync.signal = cnt(l, 3); u.tl = tl(l, 3);
    CL_LAUNCH(launch_gemv(gemv_variant_, EPI_GATEUP, true, u, stream_, use_pdl_, &nc));
    prev_cnt = cnt(l, 3); prev_n = nc;
    // (5) down projection + residual
    GemvArgs w;
    w.slots = d_slots_; w.batch = B; w.pdl_early = pdl_early_;
    w.W = L.wdown; w.N = d; w.K = F; w.x = d_act_; w.x_stride = F; w.y = d_h_; w.resid = d_h_; w.y_stride = d;
    w.sync.wait = prev_cnt; w.sync.n_wait = (unsigned)prev_n; w.sync.signal = cnt(l, 4); w.tl = tl(l, 4);
    CL_LAUNCH(launch_gemv(gemv_variant_, EPI_RESID, false, w, stream_, use_pdl_, &nc));
    prev_cnt = cnt(l, 4); prev_n = nc;
  }
  if (probe_ev_) cudaEventRecord(probe_ev_[probe_idx_ + 1], stream_);
  GemvArgs lm;
  lm.slots = d_slots_; lm.batch = B; lm.pdl_early = pdl_early_;
  lm.W = lm_head_; lm.N = cfg.vocab_size; lm.K = d; lm.h = d_h_; lm.gain = final_norm_; lm.eps = cfg.rms_eps;
  lm.y = d_logits_; lm.x_stride = d; lm.y_stride = cfg.vocab_size;
  lm.sync.wait = prev_cnt; lm.sync.n_wait = (unsigned)prev_n; lm.tl = tl(L_, 0);
  CL_LAUNCH(launch_gemv(gemv_variant_, EPI_STORE, true, lm, stream_, use_pdl_ && !mega));
  if (tail) {
    StepTailArgs t;
    t.logits = d_logits_; t.vocab = cfg.vocab_size; t.tok = d_tok_; t.pos = d_pos_; t.ids_ring = d_ids_ring_;
    t.step_counter = d_step_counter_; t.ring_steps = ring_steps_; t.ring_stride = max_batch_;
    t.part_val = d_tail_val_; t.part_idx = d_tail_idx_; t.counters = d_tail_cnt_; t.slots = d_slots_; t.batch = B;
    t.sync_counters = d_sync_; t.n_sync_counters = n_sync_;
    CL_LAUNCH(launch_step_tail(t, stream_));
  }
#undef CL_LAUNCH
  return n;
}

// ---- batched token step (B >= 2): tensor-core projections (tcgen05, split-K) + per-sequence glue -----
// split-K count of a batched-decode projection: the launch is as slow as its busiest CTA, i.e.
// rounds(= ceil(tiles * s / SMs)) x k-blocks per unit.  224 gate|up tiles on 148 SMs cost 2 x 64 k-blocks unsplit but
// 8 x 13 with 5 splits (ideal 96.9); down 56 -> 50 with 9.  Among the counts within 10 % of the best the smallest wins
// (fewer partials for the consumer kernel to sum).
int pick_splits_public(int n_rows, int K) { return pick_splits(n_rows, K); }
static int pick_splits(int n_rows, int K) {
  const int tiles = (n_rows + 127) / 128, nkb = (K + 63) / 64, sms = sm_count();
  int best_cost = 1 << 30;
  int cost_of[17];
  for (int s = 1; s <= 16; ++s) {
    const int kbp = (nkb + s - 1) / s;
    cost_of[s] = -1;
    if ((nkb + kbp - 1) / kbp != s) continue;                 // every split must own >= 1 k-block
    cost_of[s] = ((tiles * s + sms - 1) / sms) * kbp;
    best_cost = std::min(best_cost, cost_of[s]);
  }
  for (int s = 1; s <= 16; ++s)
    if (cost_of[s] >= 0 && cost_of[s] * 10 <= best_cost * 11) return s;
  return 1;
}

// ---- batched token step as ONE persistent kernel (decode_mega_batch.cu): embed -> kernel (all layers + LM head) -> tail
int Engine::enqueue_step_batch_mega(int B) {
  int n = 0, r;
#define CL_LAUNCH(call) do { r = (call); if (r < 0) { set_last_error(std::string(#call) + ": " + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; } n += r; } while (0)
  const int d = cfg.d_model, F = cfg.d_ff, V = cfg.vocab_size;
  CL_LAUNCH(launch_embed(embed_, d, d_tok_, d_h_, d, d_slots_, B, stream_));
  BatchMegaArgs m;
  m.layers = d_bm_layers_; m.wmaps = d_bm_wmaps_; m.n_layers = cfg.n_layers; m.B = B; m.n_kv = cfg.n_kv_heads;
  m.nsplit = std::max(1, std::min(std::min(nsplit_, 32), sm_count() / (cfg.n_kv_heads * B)));
  m.q_dim = q_dim_; m.qkv_dim = qkv_dim_; m.vocab = V;
  m.s_qkv = pick_splits(qkv_dim_, d); m.s_o = pick_splits(d, q_dim_); m.s_gu = pick_splits(2 * F, d); m.s_dn = pick_splits(d, F);
  m.eps = cfg.rms_eps; m.rope = rope_; m.pos = d_pos_; m.block_tables = d_bt_; m.bt_stride = max_pages_per_seq_; m.slots = d_slots_;
  m.h = d_h_; m.xn = bws_->xn; m.attn = bws_->attn; m.act = bws_->act; m.part = bws_->part; m.att_part = d_attn_part_; m.att_cnt = d_attn_cnt_;
  m.logits = d_logits_; m.final_norm = final_norm_; m.bars = d_sync_;
  m.kv_layer_rows = (long long)n_pages_ * cfg.n_kv_heads * page_size_;
  m.tl = d_timeline_;
  m.max_flight = env_int("CL_BMEGA_MAX_FLIGHT", 4); m.pause_in_barrier = env_int("CL_BMEGA_PAUSE", 1);
  m.map_xn = bm_map_xn_; m.map_attn = bm_map_attn_; m.map_act = bm_map_act_; m.kmap = kmap_; m.vmap = vmap_;
  CL_LAUNCH(launch_decode_mega_batch(m, stream_));
  CL_LAUNCH(launch_gemm_bf16(bws_->xn, lm_head_, bws_->logits, nullptr, B, V, d, stream_, 1, false));
  CL_LAUNCH(launch_batch_scatter_rows(bws_->logits, V, d_logits_, V, d_slots_, B, stream_));
  StepTailArgs t;
  t.logits = d_logits_; t.vocab = V; t.tok = d_tok_; t.pos = d_pos_; t.ids_ring = d_ids_ring_;
  t.step_counter = d_step_counter_; t.ring_steps = ring_steps_; t.ring_stride = max_batch_;
  t.part_val = d_tail_val_; t.part_idx = d_tail_idx_; t.counters = d_tail_cnt_; t.slots = d_slots_; t.batch = B;
  t.sync_counters = d_sync_; t.n_sync_counters = n_sync_;
  CL_LAUNCH(launch_step_tail(t, stream_));
#undef CL_LAUNCH
  return n;
}

int Engine::enqueue_step_batched(int B) {
  const int d = cfg.d_model, F = cfg.d_ff, L_ = cfg.n_layers, V = cfg.vocab_size;
  int n = 0, r;
  // CL_STEP_PROFILE=1 (eager launches only, CL_GRAPH=0): a CUDA event after every launch; per-kernel-class device time of
  // the step — gap before the kernel included — goes to stderr
  const bool prof_env = env_int("CL_STEP_PROFILE", 0) != 0;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  cudaStreamIsCapturing(stream_, &cap);
  const bool prof = prof_env && cap == cudaStreamCaptureStatusNone;
  std::vector<cudaEvent_t> pev;
  std::vector<const char*> pname;
  auto mark = [&](const char* name) {
    if (!prof) return;
    cudaEvent_t e;
    cudaEventCreate(&e);
    cudaEventRecord(e, stream_);
    pev.push_back(e);
    pname.push_back(name);
  };
  mark("start");
#define CL_LAUNCH(call) do { r = (call); if (r < 0) { set_last_error(std::string(#call) + ": " + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; } n += r; mark(#call); } while (0)
  BatchWs& w = *bws_;
  static const int batch_attn_ctas = env_int("CL_BATCH_ATTN_CTAS", sm_count());
  static const bool bpdl_env = env_int("CL_BATCH_PDL", 1) != 0;
  const bool bp = bpdl_env && use_pdl_;   // programmatic dependent launch between the kernels of the batched step
  const int s_qkv = pick_splits(qkv_dim_, d), s_o = pick_splits(d, q_dim_), s_gu = pick_splits(2 * F, d), s_dn = pick_splits(d, F);
  CL_LAUNCH(launch_embed(embed_, d, d_tok_, d_h_, d, d_slots_, B, stream_));
  const float* pending = nullptr;   // split-K partials of the previous residual projection, folded into the next norm
  int pending_s = 0;
  for (int l = 0; l < L_; ++l) {
    const auto& L = layers_[l];
    CL_LAUNCH(launch_batch_resid_norm(d_h_, d, pending, pending_s, B, L.attn_norm, cfg.rms_eps, w.xn, d_slots_, stream_, bp));
    CL_LAUNCH(launch_gemm_bf16(w.xn, L.wqkv, w.part, nullptr, B, qkv_dim_, d, stream_, s_qkv, bp));
    QkvEpi e;
    e.rope = rope_; e.pos = d_pos_; e.block_tables = d_bt_; e.bt_stride = max_pages_per_seq_;
    e.kpool = kpool_ + (size_t)l * kv_layer_elems_; e.vpool = vpool_ + (size_t)l * kv_layer_elems_;
    e.n_heads = cfg.n_heads; e.n_kv = cfg.n_kv_heads; e.head_dim = cfg.head_dim; e.page_size = page_size_;
    CL_LAUNCH(launch_batch_rope_append(w.part, s_qkv, B, e, d_q_, q_dim_, d_slots_, stream_, bp));
    AttnDecodeArgs a;
    a.q = d_q_; a.q_stride = q_dim_;
    a.kpool = e.kpool; a.vpool = e.vpool; a.block_tables = d_bt_; a.bt_stride = max_pages_per_seq_; a.pos = d_pos_;
    a.out = d_attn_; a.out_stride = q_dim_; a.out_bf16 = w.attn; a.part = d_attn_part_; a.counters = d_attn_cnt_;   // bf16 copy = X of the o-projection
    a.slots = d_slots_; a.batch = B; a.n_heads = cfg.n_heads; a.n_kv = cfg.n_kv_heads; a.head_dim = cfg.head_dim;
    // many sequences already fill the machine: fewer KV splits per sequence (cheaper combine, fewer CTAs)
    a.page_size = page_size_; a.pdl_early = bp ? 1 : 0;
    attn_decode_tc_plan(cfg.n_kv_heads, B, nsplit_, batch_attn_ctas, &a.nsplit, &a.tc_small);
    static const bool attn_tc = env_int("CL_BATCH_ATTN_TC", 1) != 0;
    if (attn_tc && have_kv_maps_ && attn_decode_tc_supported(cfg.n_heads, cfg.n_kv_heads, cfg.head_dim, page_size_, a.nsplit))
      CL_LAUNCH(launch_attn_decode_tc(a, kmap_, vmap_, (long long)l * n_pages_ * cfg.n_kv_heads * page_size_, stream_, bp));
    else
      CL_LAUNCH(launch_attn_decode(a, stream_, bp));
    CL_LAUNCH(launch_gemm_bf16(w.attn, L.wo, w.part, nullptr, B, d, q_dim_, stream_, s_o, bp));
    CL_LAUNCH(launch_batch_resid_norm(d_h_, d, w.part, s_o, B, L.ffn_norm, cfg.rms_eps, w.xn, d_slots_, stream_, bp));
    CL_LAUNCH(launch_gemm_bf16(w.xn, L.wgu, w.part, nullptr, B, 2 * F, d, stream_, s_gu, bp));
    CL_LAUNCH(launch_batch_silu(w.part, s_gu, B, F, w.act, stream_, bp));
    CL_LAUNCH(launch_gemm_bf16(w.act, L.wdown, w.part, nullptr, B, d, F, stream_, s_dn, bp));
    pending = w.part; pending_s = s_dn;
  }
  CL_LAUNCH(launch_batch_resid_norm(d_h_, d, pending, pending_s, B, final_norm_, cfg.rms_eps, w.xn, d_slots_, stream_, bp));
  CL_LAUNCH(launch_gemm_bf16(w.xn, lm_head_, w.logits, nullptr, B, V, d, stream_, 1, bp));
  CL_LAUNCH(launch_batch_scatter_rows(w.logits, V, d_logits_, V, d_slots_, B, stream_));
  StepTailArgs t;
  t.logits = d_logits_; t.vocab = V; t.tok = d_tok_; t.pos = d_pos_; t.ids_ring = d_ids_ring_;
  t.step_counter = d_step_counter_; t.ring_steps = ring_steps_; t.ring_stride = max_batch_;
  t.part_val = d_tail_val_; t.part_idx = d_tail_idx_; t.counters = d_tail_cnt_; t.slots = d_slots_; t.batch = B;
  t.sync_counters = d_sync_; t.n_sync_counters = n_sync_;
  CL_LAUNCH(launch_step_tail(t, stream_));
#undef CL_LAUNCH
  if (prof && pev.size() > 1) {
    cudaStreamSynchronize(stream_);
    std::map<std::string, std::pair<double, int>> acc;
    double total = 0.0;
    for (size_t i = 1; i < pev.size(); ++i) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, pev[i - 1], pev[i]);
      const std::string full(pname[i]);
      std::string key = full.substr(0, full.find('('));
      if (key == "launch_gemm_bf16")
        key += full.find("L.wqkv") != std::string::npos ? ":qkv" : full.find("L.wo") != std::string::npos ? ":o" : full.find("L.wgu") != std::string::npos ? ":gate|up"
               : full.find("lm_head_") != std::string::npos ? ":lm_head" : ":down";
      acc[key].first += ms; acc[key].second += 1;
      total += ms;
    }
    fprintf(stderr, "[step profile] B=%d, %zu launches, %.3f ms on the device\n", B, pev.size() - 1, total);
    for (auto& kv : acc) fprintf(stderr, "[step profile]   %-34s n=%4d total %8.3f ms  mean %8.2f us\n", kv.first.c_str(), kv.second.second, kv.second.first, 1e3 * kv.second.first / kv.second.second);
    for (auto e : pev) cudaEventDestroy(e);
  }
  return n;
}

// Capture + instantiate + upload the step graph of batch size B (no launch).  Returns true if graphs_[B] exists afterwards.
bool Engine::ensure_graph(int B) {
  if (!use_graph_ || graph_failed_) return false;
  if (graphs_.count(B)) return true;
  for (int attempt = 0; attempt < 2; ++attempt) {
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ex = nullptr;
    cudaError_t e = cudaStreamBeginCapture(stream_, cudaStreamCaptureModeThreadLocal);
    int n = e == cudaSuccess ? enqueue_step(B, true) : -1;
    cudaError_t e2 = cudaStreamEndCapture(stream_, &g);
    if (e == cudaSuccess && n > 0 && e2 == cudaSuccess && g) e = cudaGraphInstantiate(&ex, g, 0);
    else e = cudaErrorUnknown;
    if (g) cudaGraphDestroy(g);
    if (e == cudaSuccess && ex) {
      cudaGraphUpload(ex, stream_);
      graphs_[B] = ex;
      graph_nodes_[B] = n;
      return true;
    }
    cudaGetLastError();
    if (use_pdl_) {
      fprintf(stderr, "[clengine] graph capture with PDL failed (%s); retrying without PDL\n", cudaGetErrorString(e));
      use_pdl_ = false;
    } else {
      fprintf(stderr, "[clengine] graph capture failed (%s); falling back to eager launches\n", cudaGetErrorString(e));
      graph_failed_ = true;
      break;
    }
  }
  return false;
}

// A serving engine meets every batch size 1..max_batch as requests join and leave; capturing a 32-layer step graph
// costs tens of milliseconds, which would otherwise land inside 31 separate decode steps of the first minute of traffic
// (box benchmark, 64 concurrent chats: 16.6 req/s with lazy capture against 24.6 warm).  Called once when the
// scheduler thread starts.
void Engine::precapture_graphs() {
  if (!use_graph_ || !env_int("CL_PRECAPTURE", 1)) return;
  for (int B = 1; B <= max_batch_ && !graph_failed_; ++B) ensure_graph(B);
  cudaStreamSynchronize(stream_);
}

int Engine::run_step_graph(int B) {
  if (use_graph_ && !graph_failed_) {
    ensure_graph(B);
    auto it = graphs_.find(B);
    if (it != graphs_.end()) {
      CL_CUDA_OK(cudaGraphLaunch(it->second, stream_));
      launches_ += graph_nodes_[B];
      return CL_OK;
    }
  }
  const int n = enqueue_step(B, true);
  if (n < 0) return n;
  launches_ += n;
  return CL_OK;
}

int Engine::read_logits(int slot, float* out) {
  CL_CUDA_OK(cudaMemcpyAsync(h_logits_pinned_, d_logits_ + (size_t)slot * cfg.vocab_size, (size_t)cfg.vocab_size * 4,
                             cudaMemcpyDeviceToHost, stream_));
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  memcpy(out, h_logits_pinned_, (size_t)cfg.vocab_size * 4);
  return CL_OK;
}

int Engine::set_single_slot(cl_seq_t s) {
  if (last_single_slot_ != s) {
    CL_CUDA_OK(cudaMemcpyAsync(d_slots_, &s, 4, cudaMemcpyHostToDevice, stream_));
    last_single_slot_ = s;
    slots_dirty_ = true;   // the scheduler's cached slot list no longer describes d_slots_
  }
  return CL_OK;
}

int Engine::decode_step(cl_seq_t s, int32_t id, float* logits_out, int32_t* argmax_out) {
  if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
  if (id < 0 || id >= cfg.vocab_size) { set_last_error("token id out of range"); return CL_ERR_INVALID_ARG; }
  auto& q = seqs_[s];
  int rc = ensure_capacity(s, q.len + 1);
  if (rc) return rc;
  const int hdr[2] = {id, q.len};
  CL_CUDA_OK(cudaMemcpyAsync(d_tok_ + s, &hdr[0], 4, cudaMemcpyHostToDevice, stream_));
  CL_CUDA_OK(cudaMemcpyAsync(d_pos_ + s, &hdr[1], 4, cudaMemcpyHostToDevice, stream_));
  rc = set_single_slot(s);
  if (rc) return rc;
  rc = run_step_graph(1);
  if (rc) return rc;
  q.len += 1;
  q.history.push_back(id);
  if (logits_out) { rc = read_logits(s, logits_out); if (rc) return rc; }
  if (argmax_out) {
    CL_CUDA_OK(cudaMemcpyAsync(h_ids_pinned_, d_tok_ + s, 4, cudaMemcpyDeviceToHost, stream_));
    CL_CUDA_OK(cudaStreamSynchronize(stream_));
    *argmax_out = h_ids_pinned_[0];
  } else {
    CL_CUDA_OK(cudaStreamSynchronize(stream_));
  }
  return CL_OK;
}

int Engine::prefill_tokenwise(cl_seq_t s, const int32_t* ids, int n, float* logits_out) {
  auto& q = seqs_[s];
  int rc = ensure_capacity(s, q.len + n);
  if (rc) return rc;
  CL_CUDA_OK(cudaMemcpyAsync(d_prompt_, ids, (size_t)n * 4, cudaMemcpyHostToDevice, stream_));
  CL_CUDA_OK(cudaMemcpyAsync(d_pos_ + s, &q.len, 4, cudaMemcpyHostToDevice, stream_));
  rc = set_single_slot(s);
  if (rc) return rc;
  for (int i = 0; i < n; ++i) {
    CL_CUDA_OK(cudaMemcpyAsync(d_tok_ + s, d_prompt_ + i, 4, cudaMemcpyDeviceToDevice, stream_));
    rc = run_step_graph(1);
    if (rc) return rc;
  }
  q.len += n;
  q.history.insert(q.history.end(), ids, ids + n);
  if (logits_out) return read_logits(s, logits_out);
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  return CL_OK;
}

int Engine::prefill(cl_seq_t s, const int32_t* ids, int n, float* logits_out) {
  if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
  if (n <= 0) { set_last_error("empty prompt"); return CL_ERR_INVALID_ARG; }
  for (int i = 0; i < n; ++i)
    if (ids[i] < 0 || ids[i] >= cfg.vocab_size) { set_last_error("token id out of range"); return CL_ERR_INVALID_ARG; }
  if (seqs_[s].len + n > cfg.max_seq_len) { set_last_error("sequence exceeds max_seq_len"); return CL_ERR_TOO_LONG; }
  if (n >= prefill_min_tokens_ && prefill_path_ok()) {
    // short prompts: split-K projections so that every SM streams weights (d_model <= 8192: one 1024-thread CTA per row in the glue)
    if (n <= prefill_small_max_ && cfg.d_model <= 8192 && cfg.d_model % 4 == 0) return prefill_small(s, ids, n, logits_out);
    return prefill_chunked(s, ids, n, logits_out);
  }
  return prefill_tokenwise(s, ids, n, logits_out);
}

int Engine::decode_greedy(const cl_seq_t* ss, int B, const int32_t* first_ids, int n_steps, int32_t* ids_out, float* device_ms,
                          const int* top_n, LogprobRecord* lp_out) {
  return decode_loop(ss, B, first_ids, n_steps, ids_out, device_ms, false, top_n, lp_out);
}

// n_steps batched steps on the device; with `sample`, the sampler runs after every step (slots set up by sample_setup);
// with a top_n >= 0 in top_n[0..B) (and lp_out), logprobs_kernel runs after that over all B rows (the largest top_n)
int Engine::decode_loop(const cl_seq_t* ss, int B, const int32_t* first_ids, int n_steps, int32_t* ids_out, float* device_ms,
                        bool sample, const int* top_n, LogprobRecord* lp_out) {
  if (B <= 0 || B > max_batch_ || n_steps <= 0) { set_last_error("bad batch / steps"); return CL_ERR_INVALID_ARG; }
  int lp_n = -1;
  for (int b = 0; top_n && lp_out && b < B; ++b) {
    if (top_n[b] > CL_MAX_TOP_LOGPROBS) { set_last_error("top_n above CL_MAX_TOP_LOGPROBS"); return CL_ERR_INVALID_ARG; }
    lp_n = std::max(lp_n, top_n[b]);
  }
  if (lp_n >= 0) {
    const int rc = ensure_logprobs();
    if (rc) return rc;
  }
  for (int b = 0; b < B; ++b) {
    const int s = ss[b];
    if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
    for (int c = 0; c < b; ++c) if (ss[c] == s) { set_last_error("duplicate sequence in batch"); return CL_ERR_INVALID_ARG; }
    if (first_ids[b] < 0 || first_ids[b] >= cfg.vocab_size) { set_last_error("token id out of range"); return CL_ERR_INVALID_ARG; }
    const int rc = ensure_capacity(s, seqs_[s].len + n_steps);
    if (rc) return rc;
  }
  for (int b = 0; b < B; ++b) {
    const int s = ss[b];
    CL_CUDA_OK(cudaMemcpyAsync(d_tok_ + s, &first_ids[b], 4, cudaMemcpyHostToDevice, stream_));
    CL_CUDA_OK(cudaMemcpyAsync(d_pos_ + s, &seqs_[s].len, 4, cudaMemcpyHostToDevice, stream_));
  }
  CL_CUDA_OK(cudaMemcpyAsync(d_slots_, ss, (size_t)B * 4, cudaMemcpyHostToDevice, stream_));
  last_single_slot_ = B == 1 ? ss[0] : -1;
  slots_dirty_ = true;
  float total_ms = 0.f;
  for (int done = 0; done < n_steps;) {
    const int chunk = std::min(ring_steps_, n_steps - done);
    CL_CUDA_OK(cudaMemsetAsync(d_step_counter_, 0, 4, stream_));
    CL_CUDA_OK(cudaEventRecord(ev0_, stream_));
    for (int i = 0; i < chunk; ++i) {
      int rc = run_step_graph(B);
      if (rc == CL_OK && sample) rc = launch_sampler(B, d_slots_, true);
      if (rc == CL_OK && lp_n >= 0) rc = launch_logprobs(B, d_slots_, true, lp_n);
      if (rc) return rc;
    }
    CL_CUDA_OK(cudaEventRecord(ev1_, stream_));
    CL_CUDA_OK(cudaMemcpyAsync(h_ids_pinned_, d_ids_ring_, (size_t)chunk * max_batch_ * 4, cudaMemcpyDeviceToHost, stream_));
    if (lp_n >= 0)   // the B entries of each ring row
      CL_CUDA_OK(cudaMemcpy2DAsync(h_lp_ring_, (size_t)B * sizeof(LogprobRecord), d_lp_ring_, (size_t)max_batch_ * sizeof(LogprobRecord),
                                   (size_t)B * sizeof(LogprobRecord), (size_t)chunk, cudaMemcpyDeviceToHost, stream_));
    CL_CUDA_OK(cudaStreamSynchronize(stream_));
    float ms = 0.f;
    CL_CUDA_OK(cudaEventElapsedTime(&ms, ev0_, ev1_));
    total_ms += ms;
    for (int i = 0; i < chunk; ++i)
      for (int b = 0; b < B; ++b) ids_out[(size_t)(done + i) * B + b] = h_ids_pinned_[(size_t)i * max_batch_ + b];
    if (lp_n >= 0) memcpy(lp_out + (size_t)done * B, h_lp_ring_, (size_t)chunk * B * sizeof(LogprobRecord));
    done += chunk;
  }
  for (int b = 0; b < B; ++b) {
    auto& q = seqs_[ss[b]];
    q.history.push_back(first_ids[b]);
    for (int i = 0; i + 1 < n_steps; ++i) q.history.push_back(ids_out[(size_t)i * B + b]);
    q.len += n_steps;
  }
  tokens_generated_ += (int64_t)n_steps * B;
  if (total_ms > 0.f) {
    const double tps = (double)n_steps * max_batch_ / (total_ms * 1e-3);   // capacity: steps/s x max_batch
    tok_per_sec_ewma_ = tok_per_sec_ewma_ == 0.0 ? tps : 0.8 * tok_per_sec_ewma_ + 0.2 * tps;
  }
  if (device_ms) *device_ms = total_ms;
  return CL_OK;
}

// ---- device sampler (sample_kernels.cu) -------------------------------------------------------------
bool Engine::sample_qualifies(const cl_sampling& sp, int vocab) {
  const bool penalty = sp.repeat_penalty != 1.0f && sp.repeat_last_n != 0;
  return sp.temperature > 0.f && sp.top_k >= 1 && sp.top_k <= CL_SAMPLE_MAX_TOP_K && sp.top_k < vocab &&
         (!penalty || (sp.repeat_last_n > 0 && sp.repeat_last_n <= CL_SAMPLE_MAX_WINDOW));
}

SampleSlot Engine::sample_slot(const cl_sampling& sp, int vocab, const int32_t* hist, int n_hist, uint64_t step) {
  SampleSlot h;
  if (!sample_qualifies(sp, vocab)) return h;
  h.temperature = sp.temperature; h.top_p = sp.top_p; h.penalty = sp.repeat_penalty; h.top_k = sp.top_k;
  h.seed = sp.seed; h.step = step;
  if (sp.repeat_penalty != 1.0f && sp.repeat_last_n != 0) {
    h.win_len = sp.repeat_last_n;   // an empty history leaves the window to fill with the drawn ids
    h.win_count = hist ? std::min(std::max(n_hist, 0), h.win_len) : 0;
    for (int j = 0; j < h.win_count; ++j) h.win[j] = hist[n_hist - h.win_count + j];
  }
  return h;
}

int Engine::sample_setup(cl_seq_t s, const cl_sampling& sp, const int32_t* hist, int n_hist, uint64_t step) {
  if (!d_sample_state_) { set_last_error("vocabulary too large for the device sampler"); return CL_ERR_INVALID_ARG; }
  const SampleSlot h = sample_slot(sp, cfg.vocab_size, hist, n_hist, step);
  CL_CUDA_OK(cudaMemcpyAsync(d_sample_state_ + s, &h, sizeof h, cudaMemcpyHostToDevice, stream_));
  return CL_OK;
}

int Engine::launch_sampler(int B, const int* d_slots, bool ring) {
  SampleArgs a;
  a.logits = d_logits_; a.vocab = cfg.vocab_size; a.state = d_sample_state_; a.tok = d_tok_;
  if (ring) { a.ids_ring = d_ids_ring_; a.step_counter = d_step_counter_; a.ring_steps = ring_steps_; a.ring_stride = max_batch_; }
  a.part = d_sample_part_; a.counters = d_sample_cnt_; a.slots = d_slots; a.batch = B; a.nblk = sample_nblk_;
  const int n = launch_sample(a, stream_);
  if (n < 0) { set_last_error(std::string("launch_sample: ") + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; }
  launches_ += n;
  return CL_OK;
}

int Engine::sample_slots(const cl_seq_t* ss, int n, int32_t* ids_out) {
  if (n <= 0) return CL_OK;
  if (!d_sample_state_ || n > max_seqs_) { set_last_error("sample_slots: bad slot list"); return CL_ERR_INVALID_ARG; }
  CL_CUDA_OK(cudaMemcpyAsync(d_sample_slots_, ss, (size_t)n * 4, cudaMemcpyHostToDevice, stream_));
  int rc = launch_sampler(n, d_sample_slots_, false);
  if (rc || !ids_out) return rc;
  CL_CUDA_OK(cudaMemcpyAsync(h_ids_pinned_, d_tok_, (size_t)max_seqs_ * 4, cudaMemcpyDeviceToHost, stream_));
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  for (int i = 0; i < n; ++i) ids_out[i] = h_ids_pinned_[ss[i]];
  return CL_OK;
}

int Engine::decode_sample(const cl_seq_t* ss, int B, const int32_t* first_ids, const cl_sampling* sps, const uint64_t* first_steps,
                          int n_steps, int32_t* ids_out, float* device_ms, const int* top_n, LogprobRecord* lp_out) {
  if (B <= 0 || B > max_batch_ || n_steps <= 0) { set_last_error("bad batch / steps"); return CL_ERR_INVALID_ARG; }
  if (!d_sample_state_) { set_last_error("vocabulary too large for the device sampler"); return CL_ERR_INVALID_ARG; }
  bool any = false;
  for (int b = 0; b < B; ++b) {
    const int s = ss[b];
    if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
    if (sps[b].temperature > 0.f && !sample_qualifies(sps[b], cfg.vocab_size)) {
      set_last_error("sampling options outside the device sampler's limits (CL_SAMPLE_MAX_TOP_K / CL_SAMPLE_MAX_WINDOW)");
      return CL_ERR_INVALID_ARG;
    }
    any = any || sps[b].temperature > 0.f;
  }
  std::vector<int32_t> hist;
  for (int b = 0; b < B; ++b) {
    if (first_ids[b] < 0 || first_ids[b] >= cfg.vocab_size) break;   // decode_loop reports it
    const auto& h = seqs_[ss[b]].history;
    const size_t keep = std::min<size_t>(h.size(), CL_SAMPLE_MAX_WINDOW);
    hist.assign(h.end() - keep, h.end());
    hist.push_back(first_ids[b]);
    const int rc = sample_setup(ss[b], sps[b], hist.data(), (int)hist.size(), first_steps[b]);
    if (rc) return rc;
  }
  return decode_loop(ss, B, first_ids, n_steps, ids_out, device_ms, any, top_n, lp_out);
}

// ---- log-probabilities (logprobs_kernel in sample_kernels.cu) ----------------------------------------
// Allocated by the first request that asks: an engine that never sees one holds none of it (the ring alone is 21 MB at
// max_batch 128).
int Engine::ensure_logprobs() {
  if (d_lp_rec_) return CL_OK;
  const int nblk = logprob_blocks(cfg.vocab_size);
  if (!nblk) { set_last_error("vocabulary too large for logprobs_kernel"); return CL_ERR_INVALID_ARG; }
  const size_t S = (size_t)max_seqs_, ring = (size_t)ring_steps_ * max_batch_;
  DMALLOC(d_lp_ring_, ring * sizeof(LogprobRecord));
  DMALLOC(d_lp_part_, S * nblk * CL_MAX_TOP_LOGPROBS * sizeof(unsigned long long));
  DMALLOC(d_lp_stat_, S * nblk * sizeof(float2));
  DMALLOC(d_lp_cnt_, S * 4);
  DMALLOC(d_lp_slots_, S * 4);
  CL_CUDA_OK(cudaMemsetAsync(d_lp_cnt_, 0, S * 4, stream_));
  CL_CUDA_OK(cudaMallocHost(&h_lp_rec_, S * sizeof(LogprobRecord)));
  CL_CUDA_OK(cudaMallocHost(&h_lp_ring_, ring * sizeof(LogprobRecord)));
  DMALLOC(d_lp_rec_, S * sizeof(LogprobRecord));   // last: its presence marks the set-up as complete
  return CL_OK;
}

int Engine::launch_logprobs(int B, const int* d_slots, bool ring, int top_n) {
  LogprobArgs a;
  a.logits = d_logits_; a.vocab = cfg.vocab_size; a.tok = d_tok_; a.rec = d_lp_rec_;
  if (ring) { a.rec_ring = d_lp_ring_; a.step_counter = d_step_counter_; a.ring_steps = ring_steps_; a.ring_stride = max_batch_; }
  a.part = d_lp_part_; a.stat = d_lp_stat_; a.counters = d_lp_cnt_; a.slots = d_slots; a.batch = B;
  a.nblk = logprob_blocks(cfg.vocab_size); a.top_n = top_n;
  const int n = ::cl::launch_logprobs(a, stream_);
  if (n < 0) { set_last_error(std::string("launch_logprobs: ") + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; }
  launches_ += n;
  return CL_OK;
}

int Engine::logprobs_enqueue(const cl_seq_t* ss, int n, int top_n) {
  if (n <= 0) return CL_OK;
  if (n > max_seqs_ || top_n < 0 || top_n > CL_MAX_TOP_LOGPROBS) { set_last_error("logprobs_enqueue: bad slot list"); return CL_ERR_INVALID_ARG; }
  int rc = ensure_logprobs();
  if (rc) return rc;
  if (lp_last_slots_.size() != (size_t)n || !std::equal(ss, ss + n, lp_last_slots_.begin())) {   // steady batches upload nothing
    lp_last_slots_.assign(ss, ss + n);
    CL_CUDA_OK(cudaMemcpyAsync(d_lp_slots_, lp_last_slots_.data(), (size_t)n * 4, cudaMemcpyHostToDevice, stream_));
  }
  rc = launch_logprobs(n, d_lp_slots_, false, top_n);
  if (rc) return rc;
  const int lo = *std::min_element(ss, ss + n), hi = *std::max_element(ss, ss + n);
  CL_CUDA_OK(cudaMemcpyAsync(h_lp_rec_ + lo, d_lp_rec_ + lo, (size_t)(hi - lo + 1) * sizeof(LogprobRecord), cudaMemcpyDeviceToHost, stream_));
  return CL_OK;
}

int Engine::logprobs_read(const cl_seq_t* ss, int n, int top_n, LogprobRecord* out) {
  const int rc = logprobs_enqueue(ss, n, top_n);
  if (rc) return rc;
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  for (int i = 0; i < n; ++i) out[i] = h_lp_rec_[ss[i]];
  return CL_OK;
}

// ---- parity / benchmark aids ------------------------------------------------------------------------
int Engine::seq_fake_fill(cl_seq_t s, int n_tokens) {
  if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
  if (n_tokens < 0) { set_last_error("fake_fill: negative length"); return CL_ERR_INVALID_ARG; }
  int rc = ensure_capacity(s, std::max(n_tokens, 1));
  if (rc) return rc;
  const int n = launch_fake_fill_kv(kpool_, vpool_, kv_layer_elems_, cfg.n_layers, d_bt_ + (size_t)s * max_pages_per_seq_, page_size_,
                                    cfg.n_kv_heads, cfg.head_dim, n_tokens, stream_);
  if (n < 0) { set_last_error(std::string("fake_fill: ") + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; }
  launches_ += n;
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  seqs_[s].len = n_tokens;
  seqs_[s].history.assign((size_t)n_tokens, 0);
  return CL_OK;
}

int Engine::debug_kv(cl_seq_t s, int layer, int which, int t0, int n, float* out) {
  if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
  if (layer < 0 || layer >= cfg.n_layers || t0 < 0 || n <= 0 || t0 + n > seqs_[s].len || !out) { set_last_error("debug_kv: bad range"); return CL_ERR_INVALID_ARG; }
  float* tmp = nullptr;
  const size_t bytes = (size_t)n * kv_dim_ * 4;
  CL_CUDA_OK(cudaMalloc(&tmp, bytes));
  const __nv_bfloat16* pool = (which ? vpool_ : kpool_) + (size_t)layer * kv_layer_elems_;
  int rc = CL_OK;
  if (launch_gather_kv(pool, d_bt_ + (size_t)s * max_pages_per_seq_, page_size_, cfg.n_kv_heads, cfg.head_dim, t0, n, tmp, stream_) < 0 ||
      cudaMemcpyAsync(out, tmp, bytes, cudaMemcpyDeviceToHost, stream_) != cudaSuccess || cudaStreamSynchronize(stream_) != cudaSuccess) {
    set_last_error(std::string("debug_kv: ") + cudaGetErrorString(cudaGetLastError()));
    rc = CL_ERR_CUDA;
  }
  cudaFree(tmp);
  return rc;
}

// one batched step with caller-chosen input tokens (teacher forcing); logits_out [n_seqs][vocab] (may be NULL)
int Engine::decode_step_batch(const cl_seq_t* ss, int B, const int32_t* ids, float* logits_out, int32_t* argmax_out) {
  if (B <= 0 || B > max_batch_) { set_last_error("bad batch"); return CL_ERR_INVALID_ARG; }
  for (int b = 0; b < B; ++b) {
    const int s = ss[b];
    if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
    for (int c = 0; c < b; ++c) if (ss[c] == s) { set_last_error("duplicate sequence in batch"); return CL_ERR_INVALID_ARG; }
    if (ids[b] < 0 || ids[b] >= cfg.vocab_size) { set_last_error("token id out of range"); return CL_ERR_INVALID_ARG; }
    const int rc = ensure_capacity(s, seqs_[s].len + 1);
    if (rc) return rc;
  }
  for (int b = 0; b < B; ++b) {
    const int s = ss[b];
    CL_CUDA_OK(cudaMemcpyAsync(d_tok_ + s, &ids[b], 4, cudaMemcpyHostToDevice, stream_));
    CL_CUDA_OK(cudaMemcpyAsync(d_pos_ + s, &seqs_[s].len, 4, cudaMemcpyHostToDevice, stream_));
  }
  CL_CUDA_OK(cudaMemcpyAsync(d_slots_, ss, (size_t)B * 4, cudaMemcpyHostToDevice, stream_));
  last_single_slot_ = B == 1 ? ss[0] : -1;
  slots_dirty_ = true;
  const int rc = run_step_graph(B);
  if (rc) return rc;
  for (int b = 0; b < B; ++b) {
    auto& q = seqs_[ss[b]];
    q.len += 1;
    q.history.push_back(ids[b]);
    if (logits_out) { const int r2 = read_logits(ss[b], logits_out + (size_t)b * cfg.vocab_size); if (r2) return r2; }
  }
  if (argmax_out) {
    CL_CUDA_OK(cudaMemcpyAsync(h_ids_pinned_, d_tok_, (size_t)max_seqs_ * 4, cudaMemcpyDeviceToHost, stream_));
    CL_CUDA_OK(cudaStreamSynchronize(stream_));
    for (int b = 0; b < B; ++b) argmax_out[b] = h_ids_pinned_[ss[b]];
  } else {
    CL_CUDA_OK(cudaStreamSynchronize(stream_));
  }
  return CL_OK;
}

// bench.py's roofline.dominant_kernel: n_steps single-sequence greedy steps launched eagerly (the same kernels the
// CUDA graph holds), with a CUDA-event pair on the launching stream around the step's dominant kernel — the persistent
// whole-stack kernel (or, on the per-op path, the stack of per-layer kernels between the embedding and the LM head).
int Engine::time_dominant_kernel(cl_seq_t s, int32_t first_id, int n_steps, float* kernel_ms, float* step_ms) {
  if (s < 0 || s >= max_seqs_ || !seqs_[s].live) return CL_ERR_BAD_SEQ;
  if (n_steps <= 0 || n_steps > 4096 || first_id < 0 || first_id >= cfg.vocab_size) { set_last_error("bad steps / token"); return CL_ERR_INVALID_ARG; }
  int rc = ensure_capacity(s, seqs_[s].len + n_steps);
  if (rc) return rc;
  CL_CUDA_OK(cudaMemcpyAsync(d_tok_ + s, &first_id, 4, cudaMemcpyHostToDevice, stream_));
  CL_CUDA_OK(cudaMemcpyAsync(d_pos_ + s, &seqs_[s].len, 4, cudaMemcpyHostToDevice, stream_));
  CL_CUDA_OK(cudaMemcpyAsync(d_slots_, &s, 4, cudaMemcpyHostToDevice, stream_));
  last_single_slot_ = s;
  slots_dirty_ = true;
  CL_CUDA_OK(cudaMemsetAsync(d_step_counter_, 0, 4, stream_));
  std::vector<cudaEvent_t> ev((size_t)2 * n_steps + 2);
  for (auto& e : ev) CL_CUDA_OK(cudaEventCreate(&e));
  probe_ev_ = ev.data();
  CL_CUDA_OK(cudaEventRecord(ev[2 * n_steps], stream_));
  for (int i = 0; i < n_steps && rc == CL_OK; ++i) {
    probe_idx_ = 2 * i;
    const int n = enqueue_step(1, true);
    if (n < 0) rc = n; else launches_ += n;
  }
  probe_ev_ = nullptr;
  if (rc == CL_OK && cudaEventRecord(ev[2 * n_steps + 1], stream_) != cudaSuccess) rc = CL_ERR_CUDA;
  if (rc == CL_OK && cudaStreamSynchronize(stream_) != cudaSuccess) { set_last_error(cudaGetErrorString(cudaGetLastError())); rc = CL_ERR_CUDA; }
  double k = 0.0;
  float ms = 0.f;
  if (rc == CL_OK) {
    for (int i = 0; i < n_steps; ++i) { cudaEventElapsedTime(&ms, ev[2 * i], ev[2 * i + 1]); k += ms; }
    cudaEventElapsedTime(&ms, ev[2 * n_steps], ev[2 * n_steps + 1]);
    if (kernel_ms) *kernel_ms = (float)(k / n_steps);
    if (step_ms) *step_ms = ms / n_steps;
    // the device advanced tok/pos itself; mirror it on the host
    CL_CUDA_OK(cudaMemcpy(h_ids_pinned_, d_ids_ring_, (size_t)std::min(n_steps, ring_steps_) * max_batch_ * 4, cudaMemcpyDeviceToHost));
    auto& q = seqs_[s];
    q.history.push_back(first_id);
    for (int i = 0; i + 1 < n_steps; ++i) q.history.push_back(i < ring_steps_ ? h_ids_pinned_[(size_t)i * max_batch_] : 0);
    q.len += n_steps;
    tokens_generated_ += n_steps;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  return rc;
}

int Engine::debug_timeline(long long* out, int n) {
  const int want = (cfg.n_layers * 5 + 1) * 4;
  if (!d_timeline_ || n < want) return CL_ERR_INVALID_ARG;
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  CL_CUDA_OK(cudaMemcpy(out, d_timeline_, (size_t)want * 8, cudaMemcpyDeviceToHost));
  return want;
}

int Engine::debug_hidden(float* out, int n) {
  if (last_single_slot_ < 0) return CL_ERR_INVALID_ARG;
  // negative n selects a last-layer intermediate of the most recent single-sequence step (diagnostics):
  // -1 = q (roped), -2 = attention output, -3 = SwiGLU activation
  if (n < 0) {
    const float* src = n == -1 ? d_q_ + (size_t)last_single_slot_ * q_dim_ : n == -2 ? d_attn_ + (size_t)last_single_slot_ * q_dim_
                                                                              : d_act_ + (size_t)last_single_slot_ * cfg.d_ff;
    const int cnt = n == -3 ? cfg.d_ff : q_dim_;
    CL_CUDA_OK(cudaMemcpyAsync(out, src, (size_t)cnt * 4, cudaMemcpyDeviceToHost, stream_));
    CL_CUDA_OK(cudaStreamSynchronize(stream_));
    return CL_OK;
  }
  if (n != cfg.d_model) return CL_ERR_INVALID_ARG;
  CL_CUDA_OK(cudaMemcpyAsync(out, d_h_ + (size_t)last_single_slot_ * cfg.d_model, (size_t)n * 4, cudaMemcpyDeviceToHost, stream_));
  CL_CUDA_OK(cudaStreamSynchronize(stream_));
  return CL_OK;
}

int Engine::stats(cl_stats* out) {
  memset(out, 0, sizeof *out);
  out->tokens_per_sec = capacity_tok_per_sec_;
  out->measured_tokens_per_sec = tok_per_sec_ewma_;
  int active = 0;
  for (auto& s : seqs_) active += s.live ? 1 : 0;
  out->active_seqs = active;
  {
    std::lock_guard<std::mutex> lk(q_mu_);
    out->queue_depth = (int)queue_.size();
  }
  out->load = (double)(active + out->queue_depth) / (double)max_batch_;   // queued requests count as load: > 1 = requests are waiting
  out->kv_pages_total = n_pages_;
  out->kv_pages_used = pool_ ? pool_->used_pages() : 0;
  out->tokens_generated = tokens_generated_;
  out->requests_completed = requests_completed_;
  out->preemptions = preemptions_;
  out->sched_decode_steps = sched_decode_steps_;
  out->sched_decode_ns = sched_decode_ns_;
  out->sched_prefill_calls = sched_prefill_calls_;
  out->sched_prefill_tokens = sched_prefill_tokens_;
  out->sched_prefill_ns = sched_prefill_ns_;
  out->vram_gb = vram_gb_;
  memcpy(out->gpu_model, gpu_name_, sizeof out->gpu_model);
  out->kernel_launches = launches_;
  return CL_OK;
}

}  // namespace cl
