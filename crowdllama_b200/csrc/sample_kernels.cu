// sample_kernels.cu — the device sampler: repeat penalty -> top-k -> softmax at temperature -> top-p -> one draw, for
// every sampled entry of a batch in one launch, drawing exactly the token host_util.cpp sample_token() draws.
//
// Order.  Candidates are ranked as the host's partial_sort ranks them: value descending, then id ascending.  Both are
// packed in one 64-bit key, (order-preserving bits of the value) << 32 | (0xffffffff - id), so a descending sort of
// the keys is that order and no two keys are equal.  -0 is keyed as +0 (the host compares them equal).
//
// Repeat penalty without rewriting the row.  With a window of W distinct ids, the k best after the penalty are among
// (the k + W best of the raw row that are not in the window) + (the window ids with their penalised values): a
// non-window id that ranks k-th or better after the penalty has at most k - 1 non-window ids and W window ids above
// it in the raw row.  That holds for a penalty above or below 1.
//
// Work split.  grid (nblk, batch): each CTA selects the k + W best keys of its slice of the row (<= kSampleChunk
// entries; an exact radix select narrows the slice to a few hundred entries, which are sorted in shared memory) and
// publishes them; the last CTA of the row to arrive (arrival counter, as in step_tail_kernel) merges
// the nblk lists in a fixed order, applies the penalty, selects the k best and runs the tail.  No float atomics and
// no order-dependent reduction: every run gives the same bits.
//
// Tail.  On at most CL_SAMPLE_MAX_TOP_K candidates, in double precision and in the host's operation order, with
// explicitly rounded intrinsics so that no FMA contraction can change it.  The exponentials are computed in parallel
// (each value is the same whichever thread computes it); the sums and the walk run sequentially on one thread.
#include <cstdio>

#include "common.cuh"
#include "kernels.h"

namespace cl {

namespace {

constexpr int kSampleThreads = 1024;
constexpr int kSampleChunk = 8192;   // row entries one CTA sorts (64 KiB of keys)
constexpr int kSampleFinal = 256;    // >= kSampleCand: the post-penalty candidate set, sorted once
constexpr int kSampleSmall = 2048;   // the radix filter stops once at most this many entries remain
constexpr int kSamplePerThread = kSampleChunk / kSampleThreads;

__device__ __forceinline__ uint32_t order_bits(float v) {
  uint32_t u = __float_as_uint(v);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float order_value(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}
__device__ __forceinline__ unsigned long long make_key(float v, int id) {
  return ((unsigned long long)order_bits(v) << 32) | (unsigned long long)(0xffffffffu - (uint32_t)id);
}
__device__ __forceinline__ int key_id(unsigned long long k) { return (int)(0xffffffffu - (uint32_t)k); }
__device__ __forceinline__ float key_value(unsigned long long k) { return order_value((uint32_t)(k >> 32)); }
// key 0 pads a list: it ranks below every real entry and decodes to id 0xffffffff (never < vocab)

// descending bitonic sort of n (power of two) keys in shared memory; every thread of the CTA calls it
__device__ void bitonic_desc(unsigned long long* s, int n) {
  __syncthreads();
  for (int k = 2; k <= n; k <<= 1)
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int p = threadIdx.x; p < (n >> 1); p += blockDim.x) {
        const int i = ((p & ~(j - 1)) << 1) | (p & (j - 1)), ixj = i + j;   // j is a power of two
        const unsigned long long x = s[i], y = s[ixj];
        const bool desc = (i & k) == 0;
        if (desc ? x < y : x > y) { s[i] = y; s[ixj] = x; }
      }
      __syncthreads();
    }
}

__device__ __forceinline__ int pow2_at_least(int n) {
  int p = 256;
  while (p < n) p <<= 1;
  return p;
}

struct SelectShared { int hist[256]; int count, sel, sel_above, sel_cnt; };

// s[0, M) <- the M largest keys held by the CTA's threads (kv[] == 0: no entry), in descending order (zero padded when
// there are fewer).  Exact radix select on the top 32 bits (the value's order bits), 8 bits per pass from the top, until
// at most kSampleSmall entries are at or above the selected prefix; only those are sorted.  Massive ties (e.g. a
// constant row) leave more after the last pass, and then all of them are sorted: the result is the same either way.
__device__ void top_m_sorted(const unsigned long long (&kv)[kSamplePerThread], int M, unsigned long long* s, SelectShared& sh) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) sh.count = 0;
  __syncthreads();
  int mine = 0;
#pragma unroll
  for (int q = 0; q < kSamplePerThread; ++q) mine += kv[q] != 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
  if (lane == 0 && mine) atomicAdd(&sh.count, mine);
  __syncthreads();
  uint32_t prefix = 0u, mask = 0u;
  int above = 0, cand = sh.count;                       // above: entries whose masked bits exceed the prefix
  for (int shift = 24; shift >= 0 && cand > kSampleSmall; shift -= 8) {
    for (int i = tid; i < 256; i += blockDim.x) sh.hist[i] = 0;
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kSamplePerThread; ++q) {
      const uint32_t hi = (uint32_t)(kv[q] >> 32);
      if (kv[q] && (hi & mask) == prefix) atomicAdd(&sh.hist[(hi >> shift) & 255u], 1);
    }
    __syncthreads();
    if (warp == 0) {                                     // the digit at which the count from the top reaches M - above
      const int need = M - above;
      int c[8], tot = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) { c[q] = sh.hist[lane * 8 + q]; tot += c[q]; }
      int suf = tot;                                     // entries in this lane's digits and every higher lane's
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_down_sync(0xffffffffu, suf, o);
        if (lane + o < 32) suf += v;
      }
      int cum = suf - tot;
      if (cum < need && need <= suf) {
        for (int q = 7; q >= 0; --q) {
          if (cum + c[q] >= need) { sh.sel = lane * 8 + q; sh.sel_above = cum; sh.sel_cnt = c[q]; break; }
          cum += c[q];
        }
      }
    }
    __syncthreads();
    prefix |= (uint32_t)sh.sel << shift;
    mask |= 255u << shift;
    above += sh.sel_above;
    cand = above + sh.sel_cnt;
    __syncthreads();
  }
  if (tid == 0) sh.count = 0;
  __syncthreads();
#pragma unroll
  for (int q = 0; q < kSamplePerThread; ++q)
    if (kv[q] && ((uint32_t)(kv[q] >> 32) & mask) >= prefix) s[atomicAdd(&sh.count, 1)] = kv[q];
  __syncthreads();
  const int cnt = sh.count, n = pow2_at_least(cnt);
  for (int i = cnt + tid; i < n; i += blockDim.x) s[i] = 0ull;
  bitonic_desc(s, n);                                   // the arrival order of the compaction does not matter
}

// host_util.cpp uniform01: splitmix64 finaliser of (seed * golden + step + offset), top 53 bits
__device__ __forceinline__ double uniform01(unsigned long long seed, unsigned long long step) {
  unsigned long long x = seed * 0x9E3779B97F4A7C15ull + step + 0x632BE59BD9B4E019ull;
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return __dmul_rn(__ull2double_rn(x >> 11), 1.0 / 9007199254740992.0);
}

}  // namespace

__global__ void __launch_bounds__(kSampleThreads, 1) sample_topk_kernel(const SampleArgs a) {
  extern __shared__ unsigned long long sk[];          // kSampleChunk keys
  __shared__ unsigned long long sf[kSampleFinal];
  __shared__ double sp[CL_SAMPLE_MAX_TOP_K];
  __shared__ int swin[CL_SAMPLE_MAX_WINDOW];
  __shared__ int is_last_s;
  __shared__ SelectShared sel;
  const int b = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x;
  const int slot = a.slots ? a.slots[b] : b;
  SampleSlot* st = a.state + slot;
  const int k = st->top_k;
  const float temperature = st->temperature;
  if (k <= 0 || !(temperature > 0.f)) return;        // greedy / host-sampled slot: the step tail's id stays
  const int V = a.vocab, nblk = a.nblk;
  const int L = st->win_len;
  const int nwin = L > 0 ? min(st->win_count, L) : 0;
  const int M = k + nwin;                              // candidates each CTA keeps
  const float* lg = a.logits + (size_t)slot * V;

  // ---- 1. the M best of this CTA's slice, sorted, are published
  const int C = (V + nblk - 1) / nblk, i0 = blk * C, i1 = min(V, i0 + C);
  unsigned long long kv[kSamplePerThread];
#pragma unroll
  for (int q = 0; q < kSamplePerThread; ++q) {
    const int id = i0 + q * kSampleThreads + tid;
    kv[q] = id < i1 ? make_key(__ldcs(lg + id), id) : 0ull;
  }
  top_m_sorted(kv, M, sk, sel);
  unsigned long long* part = a.part + (size_t)slot * nblk * kSampleCand;
  if (nblk > 1) {
    for (int j = tid; j < M; j += blockDim.x) part[(size_t)blk * kSampleCand + j] = sk[j];
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      const unsigned old = atomicAdd(a.counters + slot, 1u);
      is_last_s = old == (unsigned)nblk - 1;
      if (is_last_s) a.counters[slot] = 0u;
    }
    __syncthreads();
    if (!is_last_s) return;
    __threadfence();
    // ---- 2. merge: the M best of the nblk lists (fixed layout: the result does not depend on the arrival order)
#pragma unroll
    for (int q = 0; q < kSamplePerThread; ++q) {
      const int i = q * kSampleThreads + tid;
      kv[q] = i < nblk * M ? __ldcg(part + (size_t)(i / M) * kSampleCand + i % M) : 0ull;
    }
    top_m_sorted(kv, M, sk, sel);
  }

  // ---- 3. repeat penalty: drop the window ids from the M best, add them back with their penalised values
  if (tid < nwin) swin[tid] = st->win[tid];
  __syncthreads();
  if (tid < kSampleCand) {
    unsigned long long key = 0ull;
    if (tid < M) {
      key = sk[tid];
      const int id = key_id(key);
      for (int j = 0; j < nwin; ++j) if (swin[j] == id) { key = 0ull; break; }
    }
    sf[tid] = key;
  } else if (tid < kSampleFinal) {
    const int j = tid - kSampleCand;
    unsigned long long key = 0ull;
    if (j < nwin) {
      const int id = swin[j];
      bool first = id >= 0 && id < V;
      for (int q = 0; q < j && first; ++q) first = swin[q] != id;   // the host penalises each distinct id once
      if (first) {
        const float v = lg[id], p = st->penalty;
        key = make_key(v > 0.f ? __fdiv_rn(v, p) : __fmul_rn(v, p), id);
      }
    }
    sf[tid] = key;
  }
  bitonic_desc(sf, kSampleFinal);                      // sf[0, k): the k best, in the host's order

  // ---- 4. tail
  const float mx = key_value(sf[0]);
  if (tid < k) sp[tid] = exp(__ddiv_rn((double)__fsub_rn(key_value(sf[tid]), mx), (double)temperature));
  __syncthreads();
  if (tid != 0) return;
  double den = 0.0;
  for (int i = 0; i < k; ++i) den = __dadd_rn(den, sp[i]);
  int keep = k;
  const float top_p = st->top_p;
  if (top_p > 0.f && top_p < 1.f) {
    double cum = 0.0;
    for (int i = 0; i < k; ++i) {
      cum = __dadd_rn(cum, __ddiv_rn(sp[i], den));
      if (cum >= (double)top_p) { keep = i + 1; break; }
    }
  }
  double tot = 0.0;
  for (int i = 0; i < keep; ++i) tot = __dadd_rn(tot, sp[i]);
  const unsigned long long step = st->step;
  const double u = __dmul_rn(uniform01(st->seed, step), tot);
  double cum = 0.0;
  int pick = key_id(sf[keep - 1]);
  for (int i = 0; i < keep; ++i) {
    cum = __dadd_rn(cum, sp[i]);
    if (u < cum) { pick = key_id(sf[i]); break; }
  }

  // ---- 5. write-back: next input token, the ring entry of this step, the draw counter and the window
  a.tok[slot] = pick;
  if (a.ids_ring) a.ids_ring[(size_t)((*a.step_counter - 1) % a.ring_steps) * a.ring_stride + b] = pick;
  st->step = step + 1;
  if (L > 0) {
    st->win[st->win_count % L] = pick;
    st->win_count += 1;
  }
}

// ---- log-probabilities of the emitted tokens ----------------------------------------------------------------------
// Raw distribution: log_softmax of the row as the step left it.  grid (nblk, batch) over the same slices as the sampler;
// each CTA computes its slice's max m_b and s_b = sum exp(x - m_b) (per-thread sums in a fixed order, then fixed
// shuffle and shared-memory trees: no float atomics) and, with top_n > 0, the top_n best keys of the slice
// (top_m_sorted).  The last CTA of the row to arrive merges in block order: M = max m_b, S = sum_b s_b exp(m_b - M),
// lse = M + log S, and the top_n best of the nblk lists.  A row's record depends only on the row: the same bits at any
// batch size or position.  -inf entries add nothing to S and rank below every finite entry.
__global__ void __launch_bounds__(kSampleThreads, 1) logprobs_kernel(const LogprobArgs a) {
  extern __shared__ unsigned long long sk[];          // kSampleChunk keys (top_n > 0 only)
  __shared__ float red[32];
  __shared__ float lse_s;
  __shared__ int is_last_s;
  __shared__ SelectShared sel;
  const int b = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int slot = a.slots ? a.slots[b] : b;
  const int V = a.vocab, nblk = a.nblk, N = a.top_n;
  const float* lg = a.logits + (size_t)slot * V;

  // ---- 1. slice max, sum of exp(x - max), top_n keys
  const int C = (V + nblk - 1) / nblk, i0 = blk * C, i1 = min(V, i0 + C);
  float v[kSamplePerThread];
  float m = -INFINITY;
#pragma unroll
  for (int q = 0; q < kSamplePerThread; ++q) {
    const int id = i0 + q * kSampleThreads + tid;
    v[q] = id < i1 ? __ldcs(lg + id) : -INFINITY;
    m = fmaxf(m, v[q]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = red[lane];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  __syncthreads();                                     // red[] is reused for the sums
  float s = 0.f;
#pragma unroll
  for (int q = 0; q < kSamplePerThread; ++q) s += v[q] > -INFINITY ? expf(v[q] - m) : 0.f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) red[warp] = s;
  __syncthreads();
  s = red[lane];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  unsigned long long kv[kSamplePerThread];
  if (N > 0) {
#pragma unroll
    for (int q = 0; q < kSamplePerThread; ++q) {
      const int id = i0 + q * kSampleThreads + tid;
      kv[q] = id < i1 ? make_key(v[q], id) : 0ull;
    }
    top_m_sorted(kv, N, sk, sel);
  }
  if (nblk > 1) {
    unsigned long long* part = a.part + (size_t)slot * nblk * CL_MAX_TOP_LOGPROBS;
    if (tid < N) part[(size_t)blk * CL_MAX_TOP_LOGPROBS + tid] = sk[tid];
    if (tid == 0) a.stat[(size_t)slot * nblk + blk] = make_float2(m, s);
    __threadfence();
    __syncthreads();
    if (tid == 0) {
      const unsigned old = atomicAdd(a.counters + slot, 1u);
      is_last_s = old == (unsigned)nblk - 1;
      if (is_last_s) a.counters[slot] = 0u;
    }
    __syncthreads();
    if (!is_last_s) return;
    __threadfence();
    // ---- 2. merge in block order (the result does not depend on the arrival order)
    if (tid == 0) {
      const float2* st = a.stat + (size_t)slot * nblk;
      float M = -INFINITY;
      for (int j = 0; j < nblk; ++j) M = fmaxf(M, __ldcg(&st[j].x));
      float S = 0.f;
      for (int j = 0; j < nblk; ++j) {
        const float2 ms = __ldcg(st + j);
        if (ms.x > -INFINITY) S += ms.y * expf(ms.x - M);
      }
      lse_s = M + logf(S);
    }
    if (N > 0) {
#pragma unroll
      for (int q = 0; q < kSamplePerThread; ++q) {
        const int i = q * kSampleThreads + tid;
        kv[q] = i < nblk * N ? __ldcg(part + (size_t)(i / N) * CL_MAX_TOP_LOGPROBS + i % N) : 0ull;
      }
      top_m_sorted(kv, N, sk, sel);                    // ends with __syncthreads: lse_s is visible
    }
  } else if (tid == 0) {
    lse_s = m + logf(s);
  }
  __syncthreads();

  // ---- 3. the record
  const float lse = lse_s;
  LogprobRecord* r = a.rec_ring ? a.rec_ring + (size_t)((*a.step_counter - 1) % a.ring_steps) * a.ring_stride + b : a.rec + slot;
  if (tid == 0) {
    const int chosen = a.tok[slot];
    r->lse = lse;
    r->logprob = chosen >= 0 && chosen < V ? lg[chosen] - lse : -INFINITY;
  }
  if (tid < N) {
    const unsigned long long key = sk[tid];
    r->top_ids[tid] = key ? key_id(key) : -1;          // key 0: fewer than top_n entries in the row
    r->top_logprobs[tid] = key ? key_value(key) - lse : -INFINITY;
  }
}

int logprob_blocks(int vocab) {
  if (vocab <= 0) return 0;
  const int nblk = (vocab + kSampleChunk - 1) / kSampleChunk;
  if (nblk * CL_MAX_TOP_LOGPROBS > kSampleChunk) return 0;   // the merge must fit the registers of one CTA
  return nblk;
}

int launch_logprobs(const LogprobArgs& a, cudaStream_t st) {
  static PerDeviceOnce once;
  const int smem = kSampleChunk * (int)sizeof(unsigned long long);
  if (once.pending()) {
    cudaFuncSetAttribute(logprobs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    once.mark();
  }
  if (a.batch <= 0 || a.nblk <= 0 || a.nblk != logprob_blocks(a.vocab) || a.top_n < 0 || a.top_n > CL_MAX_TOP_LOGPROBS) return -1;
  logprobs_kernel<<<dim3(a.nblk, a.batch), kSampleThreads, a.top_n > 0 ? smem : 0, st>>>(a);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

int sample_blocks(int vocab) {
  if (vocab <= 0) return 0;
  const int nblk = (vocab + kSampleChunk - 1) / kSampleChunk;
  if (nblk * kSampleCand > kSampleChunk) return 0;    // the merge must fit the same shared buffer
  return nblk;
}

int launch_sample(const SampleArgs& a, cudaStream_t st) {
  static PerDeviceOnce once;
  const int smem = kSampleChunk * (int)sizeof(unsigned long long);
  if (once.pending()) {
    cudaFuncSetAttribute(sample_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    once.mark();
  }
  if (a.batch <= 0 || a.nblk <= 0 || a.nblk != sample_blocks(a.vocab)) return -1;
  sample_topk_kernel<<<dim3(a.nblk, a.batch), kSampleThreads, smem, st>>>(a);
  return cudaGetLastError() == cudaSuccess ? 1 : -1;
}

}  // namespace cl
