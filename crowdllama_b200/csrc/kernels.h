// kernels.h — host-side launch interface of the sm_100a kernels (internal to libclengine.so).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/clengine.h"

namespace cl {

// Dependencies inside the token step (common.cuh: wait_counter_warp / signal_counter).
struct StepSync {
  const unsigned* wait = nullptr;   // producer node's counter (nullptr => griddepcontrol.wait)
  unsigned n_wait = 0;              // CTAs of the producer node
  unsigned* signal = nullptr;       // this node's counter (nullptr => none)
};
// o-projection prologue: the cross-split softmax combine of the attention partials, distributed over the
// o-projection's CTAs (each combines a slice of the H*D outputs), then a grid-wide counter barrier.
struct AttnCombine {
  const float* part = nullptr;      // [slot][n_kv][nsplit][rep][head_dim + 2]  (nullptr => x is read as is)
  int nsplit = 0, n_kv = 0, rep = 0, head_dim = 0;
  float* x_out = nullptr;           // [slot][x_stride] combined, bf16-rounded attention output
  unsigned* phase = nullptr;        // counter: CTAs of THIS kernel that have written their slice
};

enum GemvEpi { EPI_STORE = 0, EPI_RESID = 1, EPI_GATEUP = 2, EPI_QKV = 3 };

// EPI_QKV: the q|k|v projection's rows are stored ROPE-PAIR-INTERLEAVED (within each head, row 2j holds
// dim j and row 2j+1 holds dim j + head_dim/2), so the row pair a GEMV thread owns is exactly one RoPE
// rotation pair: the epilogue rotates, rounds to bf16, writes q to y[slot][H*D] (natural dim order) and
// appends k / v straight into the paged cache.  The attention kernel then needs no RoPE and no append.
struct QkvEpi {
  const float2* rope = nullptr;       // [max_pos][head_dim/2]
  const int* pos = nullptr;           // [slot]
  const int* block_tables = nullptr;  // [slot][bt_stride]
  int bt_stride = 0;
  __nv_bfloat16* kpool = nullptr;     // this layer
  __nv_bfloat16* vpool = nullptr;
  int n_heads = 0, n_kv = 0, head_dim = 0, page_size = 0;
};

// y[slot] = epi(W * x[slot]).  Row pairs (2i, 2i+1) are always processed together so the
// gate/up interleaving (row 2i = gate_i, row 2i+1 = up_i) needs no special casing.
struct GemvArgs {
  const __nv_bfloat16* W = nullptr;  // [N][K] row-major
  int N = 0, K = 0;
  const float* x = nullptr;          // !norm: [slot][x_stride] bf16-rounded fp32 inputs
  const float* h = nullptr;          // norm: residual stream [slot][x_stride]
  const float* gain = nullptr;       // norm gains [K]
  float eps = 0.f;
  float* y = nullptr;                // [slot][y_stride]
  const float* resid = nullptr;      // EPI_RESID (may alias y)
  int x_stride = 0, y_stride = 0;
  const int* slots = nullptr;        // blockIdx.y = b -> slot (nullptr => identity)
  int batch = 1;
  int pdl_early = 1;                 // 1: trigger dependents at kernel start; 0: when this CTA has issued its last load
  QkvEpi qkv;                        // EPI_QKV only
  StepSync sync;
  AttnCombine comb;                  // EPI_RESID o-projection only
  long long* tl = nullptr;           // debug timeline (CL_TIMELINE=1): 4 globaltimer stamps written by CTA 0
};

struct AttnDecodeArgs {
  const float* q = nullptr;          // [slot][q_stride] roped, bf16-rounded query of the current token
  int q_stride = 0;
  const __nv_bfloat16* kpool = nullptr;  // this layer: [n_pages][n_kv][page][head_dim]; holds tokens 0..pos
  const __nv_bfloat16* vpool = nullptr;
  const int* block_tables = nullptr; // [slot][bt_stride]
  int bt_stride = 0;
  const int* pos = nullptr;          // [slot] index of the current token (context = pos + 1 tokens)
  float* out = nullptr;              // [slot][out_stride] bf16-rounded fp32
  int out_stride = 0;
  __nv_bfloat16* out_bf16 = nullptr; // optional: the same values as bf16 [batch index][out_stride] (X operand of the batched o-projection)
  float* part = nullptr;             // [slot][n_kv][nsplit][rep][head_dim + 2]
  unsigned* counters = nullptr;      // [slot][n_kv]
  const int* slots = nullptr;
  int batch = 1;
  int n_heads = 0, n_kv = 0, head_dim = 0, page_size = 0, nsplit = 0;
  int pdl_early = 1;
  StepSync sync;                     // sync.signal != nullptr: publish partials only, the consumer combines
  long long* tl = nullptr;
  int ring_bytes = 0;                // filled by the launcher
  int tc_small = 0;                  // attn_decode_tc: 4-warp CTAs, two per SM (attn_decode_tc_plan)
};

struct StepTailArgs {                // argmax over logits, advance the sequence
  const float* logits = nullptr;     // [slot][vocab]
  int vocab = 0;
  int* tok = nullptr;                // [slot] next input token (written)
  int* pos = nullptr;                // [slot] incremented
  int* ids_ring = nullptr;           // [ring_steps][max_batch] generated ids
  int* step_counter = nullptr;       // device scalar, incremented once per step
  unsigned* sync_counters = nullptr; // zeroed at the end of every step (StepSync)
  int n_sync_counters = 0;
  int ring_steps = 0, ring_stride = 0;
  float* part_val = nullptr;         // [slot][nblk]
  int* part_idx = nullptr;
  unsigned* counters = nullptr;      // [slot]
  const int* slots = nullptr;
  int batch = 1;
};

// per-slot state of the device sampler (sample_kernels.cu).  The kernel advances `step` and the window after each draw.
struct SampleSlot {
  float temperature = 0.f, top_p = 0.f, penalty = 1.f;
  int top_k = 0;                     // 0: the slot is not sampled on the device (greedy, or outside the device limits)
  int win_len = 0;                   // repeat_last_n while the penalty is on, else 0
  int win_count = 0;                 // ids appended so far: win[0, min(win_count, win_len)) hold the window, id j at j % win_len
  unsigned long long seed = 0, step = 0;
  int win[CL_SAMPLE_MAX_WINDOW] = {};
};

struct SampleArgs {
  const float* logits = nullptr;     // [slot][vocab], read in place
  int vocab = 0;
  SampleSlot* state = nullptr;       // [slot]
  int* tok = nullptr;                // [slot] next input token: overwritten for the sampled slots
  int* ids_ring = nullptr;           // [ring_steps][ring_stride] (nullptr: not written) — entry of the step just run
  const int* step_counter = nullptr; // already bumped by the step: the step's ring row is (*step_counter - 1) % ring_steps
  int ring_steps = 0, ring_stride = 0;
  unsigned long long* part = nullptr;// [slot][nblk][kSampleCand] per-CTA candidate keys
  unsigned* counters = nullptr;      // [slot] arrival counters (self re-arming)
  const int* slots = nullptr;        // [batch] (nullptr: identity)
  int batch = 1;
  int nblk = 1;                      // CTAs per row: sample_blocks(vocab)
};
constexpr int kSampleCand = CL_SAMPLE_MAX_TOP_K + CL_SAMPLE_MAX_WINDOW;   // candidates one CTA keeps for the merge
int sample_blocks(int vocab);        // CTAs per row; 0 if the vocabulary is too large for the sampler
int launch_sample(const SampleArgs& a, cudaStream_t st);

// one generated token's log-probabilities (logprobs_kernel in sample_kernels.cu; clengine.h cl_logprobs)
struct LogprobRecord {
  float lse = 0.f;                                  // logsumexp of the row
  float logprob = 0.f;                              // logits[chosen] - lse
  int top_ids[CL_MAX_TOP_LOGPROBS] = {};            // [0, top_n): value descending, then id ascending
  float top_logprobs[CL_MAX_TOP_LOGPROBS] = {};
};

struct LogprobArgs {
  const float* logits = nullptr;     // [slot][vocab], read in place
  int vocab = 0;
  const int* tok = nullptr;          // [slot] the emitted id of the row (step tail's argmax or the device sampler's draw)
  LogprobRecord* rec = nullptr;      // [slot] (used when rec_ring is nullptr)
  LogprobRecord* rec_ring = nullptr; // [ring_steps][ring_stride]: entry b of the step just run (as SampleArgs::ids_ring)
  const int* step_counter = nullptr;
  int ring_steps = 0, ring_stride = 0;
  unsigned long long* part = nullptr;// [slot][nblk][CL_MAX_TOP_LOGPROBS] per-CTA top keys
  float2* stat = nullptr;            // [slot][nblk] per-CTA (max, sum of exp(x - max))
  unsigned* counters = nullptr;      // [slot] arrival counters (self re-arming)
  const int* slots = nullptr;        // [batch] (nullptr: identity)
  int batch = 1;
  int nblk = 1;                      // CTAs per row: logprob_blocks(vocab)
  int top_n = 0;                     // 0..CL_MAX_TOP_LOGPROBS, the same for every row of the launch
};
int logprob_blocks(int vocab);       // CTAs per row; 0 if the vocabulary is too large
int launch_logprobs(const LogprobArgs& a, cudaStream_t st);

// every launcher returns the number of kernels it enqueued (for cl_stats.kernel_launches)
int launch_gemv(int variant, int epi, bool norm, const GemvArgs& a, cudaStream_t st, bool pdl, int* n_ctas = nullptr);
int launch_attn_decode(const AttnDecodeArgs& a, cudaStream_t st, bool pdl);
// tensor-core variant for the batched step (attn_decode_tc.cu): head_dim 128, 4 q heads per kv head, page 32;
// kmap / vmap = pool-wide 2-D tensor maps (make_tmap_2d_bf16, box {64, 32}), layer_row0 = first row of this layer
bool attn_decode_tc_supported(int n_heads, int n_kv, int head_dim, int page_size, int nsplit);
void attn_decode_tc_plan(int n_kv, int batch, int nsplit_max, int cta_budget, int* nsplit, int* small);   // splits + kernel shape of a batched step
int launch_attn_decode_tc(const AttnDecodeArgs& a, const CUtensorMap& kmap, const CUtensorMap& vmap, long long layer_row0, cudaStream_t st,
                          bool pdl);
int launch_embed(const __nv_bfloat16* table, int d, const int* tok, float* h, int h_stride, const int* slots,
                 int batch, cudaStream_t st);
int launch_step_tail(const StepTailArgs& a, cudaStream_t st);
// zero the step counters (run once at init; the per-step reset is part of step_bump_kernel)
int launch_zero_u32(unsigned* p, int n, cudaStream_t st);
// rope_hd > 0: rows are written rope-pair-interleaved per head of rope_hd rows (see QkvEpi)
int launch_synth_bf16(__nv_bfloat16* out, int64_t n_logical, int k_cols, int row_mult, int row_off, uint64_t seed,
                      int key, float scale, cudaStream_t st, int rope_hd = 0);
int launch_synth_gain(float* out, int n, uint64_t seed, int key, float scale, cudaStream_t st);
int launch_bf16_to_f32(const __nv_bfloat16* in, float* out, int64_t n, cudaStream_t st);
int launch_fill_u16(uint16_t* p, int64_t n, uint16_t v, cudaStream_t st);
// parity aid: the oracle's oc_seq_fake_fill pattern into tokens 0..n_tokens-1 of one sequence, all layers
int launch_fake_fill_kv(__nv_bfloat16* kpool, __nv_bfloat16* vpool, size_t layer_elems, int n_layers, const int* block_table,
                        int page_size, int n_kv, int head_dim, int n_tokens, cudaStream_t st);

int launch_gather_kv(const __nv_bfloat16* pool_layer, const int* block_table, int page_size, int n_kv, int head_dim, int t0, int n,
                     float* out, cudaStream_t st);

// ---- persistent whole-stack decode kernel (decode_mega.cu) ----------------------------------------
struct MegaLayer {
  const __nv_bfloat16* wqkv; const __nv_bfloat16* wo; const __nv_bfloat16* wgu; const __nv_bfloat16* wdown;
  const float* attn_norm; const float* ffn_norm;
  __nv_bfloat16* kpool; __nv_bfloat16* vpool;
};
struct MegaArgs {
  const MegaLayer* layers = nullptr;   // device array [n_layers]
  int n_layers = 0, q_dim = 0, qkv_dim = 0, n_heads = 0, n_kv = 0, nsplit = 0;
  float eps = 0.f;
  const float2* rope = nullptr;
  const int* pos = nullptr;
  const int* block_tables = nullptr;
  int bt_stride = 0;
  const int* slots = nullptr;          // slots[0] is the sequence slot
  float* h = nullptr;                  // [slot][d] residual stream (in: embedding, out: final hidden)
  float* q = nullptr;                  // [slot][q_dim]
  float* attn_x = nullptr;             // [slot][q_dim]
  float* act = nullptr;                // [slot][d_ff]
  float* part = nullptr;               // attention partials
  unsigned* bars = nullptr;            // [n_layers * 6] grid-barrier counters, zero at kernel start
  unsigned* tile_ctr = nullptr;        // [n_layers * 4] dynamic tile-scheduler counters, zero at kernel start
  unsigned* pf_ctr = nullptr;          // L2 lookahead frontier (one counter, zero at kernel start); nullptr = off
  int pause_in_barrier = 0;            // producer issues no new copies while the consumers sit in a grid barrier
  int max_flight = 6;                  // cap on bulk copies in flight per CTA (<= ring slots)
  int pf_min = 296, pf_budget = 0;     // lookahead window in tiles ahead of a CTA's own demand position
  long long* tl = nullptr;             // debug: [n_layers][16] globaltimer stamps of CTA tl_cta
  int tl_cta = 0;
  long long kv_layer_rows = 0;         // rows of one layer in the KV tensor maps (= n_pages * n_kv * page)
  alignas(64) CUtensorMap kmap;        // whole K pool as [L * n_pages * n_kv * page][head_dim], box {64, 32}, 128B swizzle
  alignas(64) CUtensorMap vmap;
};
bool make_tmap_2d_bf16(CUtensorMap* map, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_cols, uint32_t box_rows);
bool mega_supported(int d, int d_ff, int head_dim, int n_heads, int n_kv, int page_size, int nsplit);
bool mega_prepare_device();   // per device: shared-memory opt-in + "one CTA per SM fits" (call with the device current)
int launch_decode_mega(const MegaArgs& a, cudaStream_t st);

// ---- persistent BATCHED decode step (decode_mega_batch.cu): B = 2..32 sequences, Llama-3-8B / Mistral-7B layer shape ----
struct BatchMegaLayer { const float* attn_norm; const float* ffn_norm; __nv_bfloat16* kpool; __nv_bfloat16* vpool; };
struct BatchMegaArgs {
  const BatchMegaLayer* layers = nullptr;  // device array [n_layers]
  const CUtensorMap* wmaps = nullptr;      // device array [n_layers * 4 + 1]: q|k|v, o, gate|up, down per layer, then the LM head
  int n_layers = 0, B = 0, n_kv = 0, nsplit = 1, q_dim = 0, qkv_dim = 0, vocab = 0;
  int s_qkv = 1, s_o = 1, s_gu = 1, s_dn = 1;   // k splits of the four projections (engine.cu pick_splits)
  float eps = 0.f;
  const float2* rope = nullptr;
  const int* pos = nullptr;                // [slot]
  const int* block_tables = nullptr;       // [slot][bt_stride]
  int bt_stride = 0;
  const int* slots = nullptr;              // [B]
  float* h = nullptr;                      // [slot][d] residual stream
  __nv_bfloat16* xn = nullptr;             // [32][d]    normalised rows (X of q|k|v, gate|up, LM head)
  __nv_bfloat16* attn = nullptr;           // [32][q_dim] attention output (X of o)
  __nv_bfloat16* act = nullptr;            // [32][d_ff] SwiGLU activation (X of down)
  float* part = nullptr;                   // split-K partials [s][32][N]
  float* att_part = nullptr;               // attention split partials [slot][n_kv][nsplit][4][130]
  unsigned* att_cnt = nullptr;             // [slot][n_kv] self re-arming arrival counters
  float* logits = nullptr;                 // [slot][vocab]
  const float* final_norm = nullptr;
  unsigned* bars = nullptr;                // [n_layers * 8 + 1] grid-barrier counters, zero at kernel start
  long long kv_layer_rows = 0;
  int max_flight = 4;                      // 16 KB bulk copies in flight per CTA (<= ring slots); 0 = no cap
  int pause_in_barrier = 1;                // no new copy while this CTA's consumers sit in a grid barrier
  long long* tl = nullptr;                 // debug (CL_TIMELINE=1): [n_layers][16] globaltimer stamps of CTA 0 at phase ends / barrier exits
  alignas(64) CUtensorMap map_xn;          // [32][d] box {64, 32}
  alignas(64) CUtensorMap map_attn;
  alignas(64) CUtensorMap map_act;
  alignas(64) CUtensorMap kmap;            // pool-wide K / V maps, box {64, 32}
  alignas(64) CUtensorMap vmap;
};
bool batch_mega_supported(int d, int d_ff, int head_dim, int n_heads, int n_kv, int page_size, int vocab);
bool batch_mega_prepare_device();
bool make_wmap(CUtensorMap* map, const void* W, int N, int K);
int launch_decode_mega_batch(const BatchMegaArgs& a, cudaStream_t st);

bool gemv_variant_supported(int variant, int N, int K);
int sm_count();
// "done once" flag per (call site, current device): function attributes (dynamic shared memory limit, carve-out) belong to a
// device's context, so a process that opens a second GPU must set them again (ADVICE r1)
struct PerDeviceOnce {
  bool done[64] = {};
  bool* slot() { int d = 0; cudaGetDevice(&d); return &done[d & 63]; }
  bool pending() { return !*slot(); }
  void mark() { *slot() = true; }
};

// ---- prefill path (prefill_kernels.cu / gemm_tcgen05.cu) -----------------------------------------
// X bf16 [T][K] row-major, W bf16 [N][K] row-major -> Y fp32 [T][N] (+= resid when resid != nullptr)
// k_splits > 1: split-K, partial s is written to Y + s*T*N (no residual); the consumer sums the partials
int launch_gemm_bf16(const __nv_bfloat16* X, const __nv_bfloat16* W, float* Y, const float* resid, int T, int N, int K,
                     cudaStream_t st, int k_splits = 1, bool pdl = false);
bool gemm_tcgen05_supported(int T, int N, int K);
// fused prefill epilogues of the tcgen05 GEMM (gemm_tcgen05.cu): the fp32 result never leaves the SM
struct GemmEpi {
  int kind = 0;                              // 1: gate|up rows interleaved (2i gate, 2i+1 up) -> act[t][i] = bf16(silu(g) * u)
                                             // 2: q|k|v rows rope-pair-interleaved, head_dim 128 -> RoPE at pos0 + t, bf16, q_out / paged cache
  __nv_bfloat16* act = nullptr; int ld_act = 0;
  const float2* rope = nullptr; int pos0 = 0;
  __nv_bfloat16* q_out = nullptr; int q_dim = 0;
  __nv_bfloat16* kpool = nullptr; __nv_bfloat16* vpool = nullptr;   // this layer
  const int* block_table = nullptr; int page_size = 0, n_heads = 0, n_kv = 0;
};
int launch_gemm_bf16_epi(const __nv_bfloat16* X, const __nv_bfloat16* W, int T, int N, int K, const GemmEpi& epi, cudaStream_t st);
// xn[t] = bf16(rmsnorm(h[t]) * gain)
int launch_rmsnorm_bf16(const float* h, const float* gain, float eps, __nv_bfloat16* out, int T, int d, cudaStream_t st);
// rope q,k of T tokens starting at pos0; q -> bf16 [T][H][D]; k,v -> paged cache (bf16) and optional dense copies
// qkv columns arrive rope-pair-interleaved (the GEMM uses the same permuted wqkv rows)
struct RopeScatterArgs {
  const float* qkv; int qkv_stride; const float2* rope; int pos0; int T;
  __nv_bfloat16* q_out;              // [T][H*D]
  __nv_bfloat16* kpool; __nv_bfloat16* vpool; const int* block_table; int page_size;
  int n_heads, n_kv, head_dim;
  int n_split = 1; size_t split_stride = 0;   // qkv = sum of n_split split-K partials, split_stride floats apart (fixed order)
};
int launch_rope_scatter(const RopeScatterArgs& a, cudaStream_t st);
// causal attention of T new tokens (positions pos0..pos0+T-1) against the paged cache
struct AttnPrefillArgs {
  const __nv_bfloat16* q;            // [T][H*D] roped
  const __nv_bfloat16* kpool; const __nv_bfloat16* vpool; const int* block_table; int page_size;
  int pos0, T, n_heads, n_kv, head_dim;
  __nv_bfloat16* out;                // [T][H*D]
};
int launch_attn_prefill(const AttnPrefillArgs& a, cudaStream_t st);
// tcgen05 variant (attn_prefill_tc.cu): head_dim 128, page 32; kmap / vmap = pool-wide 2-D tensor maps (box {64, 32})
bool attn_prefill_tc_supported(int n_heads, int n_kv, int head_dim, int page_size, int pos0, int T);
int launch_attn_prefill_tc(const AttnPrefillArgs& a, const CUtensorMap& kmap, const CUtensorMap& vmap, long long layer_row0, cudaStream_t st);
// act = bf16(silu(gu[:, 2i]) * gu[:, 2i+1])
int launch_silu_mul_bf16(const float* gu, __nv_bfloat16* act, int T, int d_ff, cudaStream_t st);
// ---- batched decode glue (batch_kernels.cu) ------------------------------------------------------
int launch_batch_resid_norm(float* h, int d, const float* ypart, int n_split, int B, const float* gain, float eps, __nv_bfloat16* xn,
                            const int* slots, cudaStream_t st, bool pdl = false);
// xn[b] = bf16(rmsnorm(h[slots[b]]) * gain)   (PDL-aware)
int launch_batch_norm(const float* h, int d, int B, const float* gain, float eps, __nv_bfloat16* xn, const int* slots, cudaStream_t st, bool pdl);
int launch_batch_rope_append(const float* ypart, int n_split, int B, const QkvEpi& e, float* q_out, int q_stride, const int* slots,
                             cudaStream_t st, bool pdl = false);
int launch_batch_gather_bf16(const float* x, int n, int x_stride, __nv_bfloat16* xb, const int* slots, int B, cudaStream_t st);
int launch_batch_silu(const float* ypart, int n_split, int B, int d_ff, __nv_bfloat16* act, cudaStream_t st, bool pdl = false);
int launch_batch_scatter_rows(const float* y, int n, float* out, int out_stride, const int* slots, int B, cudaStream_t st);
int launch_embed_rows(const __nv_bfloat16* table, int d, const int* ids_dev, float* h, int T, cudaStream_t st);

}  // namespace cl
