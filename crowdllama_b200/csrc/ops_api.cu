// ops_api.cu — cl_op_*: single-kernel entry points of the C-ABI with HOST buffers in and out.
// Each runs exactly the kernel the token step uses (parity tests per kernel, microbenchmarks).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "engine.h"

using namespace cl;

namespace {

struct DevBuf {
  void* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
  template <typename T> T* as() { return reinterpret_cast<T*>(p); }
  cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 16); }
  cudaError_t upload(const void* h, size_t bytes) {
    cudaError_t e = alloc(bytes);
    return e != cudaSuccess ? e : cudaMemcpy(p, h, bytes, cudaMemcpyHostToDevice);
  }
};

int check_device(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device < 0 || device >= n) {
    cudaGetLastError();
    set_last_error("no CUDA device (libclengine has no CPU fallback)");
    return CL_ERR_NO_DEVICE;
  }
  CL_CUDA_OK(cudaSetDevice(device));
  return CL_OK;
}

int run_gemv(int device, int variant, int epi, bool norm, const uint16_t* w, const float* x_or_h, const float* gain, float eps,
             const float* resid, float* y, int n_rows, int k, int out_n, int iters, float* ms) {
  int rc = check_device(device);
  if (rc) return rc;
  if (!gemv_variant_supported(variant, n_rows, k)) {
    set_last_error("gemv variant does not support this shape");
    return CL_ERR_INVALID_ARG;
  }
  DevBuf dw, dx, dg, dy;
  CL_CUDA_OK(dw.upload(w, (size_t)n_rows * k * 2));
  CL_CUDA_OK(dx.upload(x_or_h, (size_t)k * 4));
  if (gain) CL_CUDA_OK(dg.upload(gain, (size_t)k * 4));
  CL_CUDA_OK(dy.alloc((size_t)std::max(out_n, n_rows) * 4));
  if (resid) CL_CUDA_OK(cudaMemcpy(dy.p, resid, (size_t)out_n * 4, cudaMemcpyHostToDevice));
  else CL_CUDA_OK(cudaMemset(dy.p, 0, (size_t)out_n * 4));
  GemvArgs a;
  a.W = dw.as<__nv_bfloat16>(); a.N = n_rows; a.K = k;
  if (norm) { a.h = dx.as<float>(); a.gain = dg.as<float>(); a.eps = eps; } else { a.x = dx.as<float>(); }
  a.y = dy.as<float>(); a.resid = resid ? dy.as<float>() : nullptr; a.x_stride = k; a.y_stride = out_n; a.batch = 1;
  cudaStream_t st = nullptr;
  if (launch_gemv(variant, epi, norm, a, st, false) < 0) { CL_CUDA_OK(cudaGetLastError()); return CL_ERR_CUDA; }
  CL_CUDA_OK(cudaDeviceSynchronize());
  CL_CUDA_OK(cudaMemcpy(y, dy.p, (size_t)out_n * 4, cudaMemcpyDeviceToHost));
  if (iters > 0 && ms && epi != EPI_RESID) {
    // timing loop: rotate over enough weight copies to exceed the 126 MB L2
    const size_t wbytes = (size_t)n_rows * k * 2;
    int copies = (int)std::min<size_t>(16, (256ull << 20) / wbytes + 1);
    std::vector<DevBuf> extra(copies > 1 ? copies - 1 : 0);
    std::vector<const __nv_bfloat16*> ws{dw.as<__nv_bfloat16>()};
    for (auto& b : extra) {
      CL_CUDA_OK(b.alloc(wbytes));
      CL_CUDA_OK(cudaMemcpy(b.p, dw.p, wbytes, cudaMemcpyDeviceToDevice));
      ws.push_back(b.as<__nv_bfloat16>());
    }
    cudaEvent_t e0, e1;
    CL_CUDA_OK(cudaEventCreate(&e0));
    CL_CUDA_OK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) { a.W = ws[i % ws.size()]; launch_gemv(variant, epi, norm, a, st, false); }
    CL_CUDA_OK(cudaDeviceSynchronize());
    CL_CUDA_OK(cudaEventRecord(e0, st));
    for (int i = 0; i < iters; ++i) { a.W = ws[i % ws.size()]; launch_gemv(variant, epi, norm, a, st, false); }
    CL_CUDA_OK(cudaEventRecord(e1, st));
    CL_CUDA_OK(cudaDeviceSynchronize());
    float t = 0.f;
    CL_CUDA_OK(cudaEventElapsedTime(&t, e0, e1));
    *ms = t / (float)iters;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
  }
  return CL_OK;
}

}  // namespace

extern "C" {

int cl_op_gemv(int device, int variant, const uint16_t* w, const float* x, float* y, int32_t n_rows, int32_t k, int32_t iters,
               float* ms) {
  if (!w || !x || !y) return CL_ERR_INVALID_ARG;
  return run_gemv(device, variant, EPI_STORE, false, w, x, nullptr, 0.f, nullptr, y, n_rows, k, n_rows, iters, ms);
}
int cl_op_gemv_residual(int device, int variant, const uint16_t* w, const float* x, const float* resid, float* y, int32_t n_rows,
                        int32_t k) {
  if (!w || !x || !y || !resid) return CL_ERR_INVALID_ARG;
  return run_gemv(device, variant, EPI_RESID, false, w, x, nullptr, 0.f, resid, y, n_rows, k, n_rows, 0, nullptr);
}
int cl_op_rmsnorm_gemv(int device, int variant, const uint16_t* w, const float* h, const float* gain, float eps, float* y,
                       int32_t n_rows, int32_t k) {
  if (!w || !h || !y || !gain) return CL_ERR_INVALID_ARG;
  return run_gemv(device, variant, EPI_STORE, true, w, h, gain, eps, nullptr, y, n_rows, k, n_rows, 0, nullptr);
}
int cl_op_rmsnorm_gateup(int device, int variant, const uint16_t* w_gu, const float* h, const float* gain, float eps, float* act,
                         int32_t d_ff, int32_t k) {
  if (!w_gu || !h || !act || !gain) return CL_ERR_INVALID_ARG;
  return run_gemv(device, variant, EPI_GATEUP, true, w_gu, h, gain, eps, nullptr, act, 2 * d_ff, k, d_ff, 0, nullptr);
}

int cl_op_attn_decode(int device, const float* q, const uint16_t* k_cache, const uint16_t* v_cache, int32_t ctx_len, int32_t n_heads,
                      int32_t n_kv, int32_t head_dim, int32_t page_size, float* out) {
  if (!q || !out || ctx_len <= 0 || !k_cache || !v_cache) return CL_ERR_INVALID_ARG;
  int rc = check_device(device);
  if (rc) return rc;
  const int rep = n_kv > 0 ? n_heads / n_kv : 0;
  if ((head_dim != 64 && head_dim != 128) || (rep != 1 && rep != 2 && rep != 4 && rep != 8) || n_heads % n_kv ||
      (page_size != 16 && page_size != 32 && page_size != 64)) {
    set_last_error("unsupported attention shape");
    return CL_ERR_INVALID_ARG;
  }
  const int P = page_size, HD = head_dim;
  const int n_pages = (ctx_len + P - 1) / P;
  // scatter the dense cache into pages in a scrambled page order (exercises the block table)
  std::vector<int> bt(n_pages);
  for (int i = 0; i < n_pages; ++i) bt[i] = (int)(((long long)i * 7 + 3) % n_pages);
  if (n_pages % 7 == 0) for (int i = 0; i < n_pages; ++i) bt[i] = n_pages - 1 - i;
  const size_t pool_elems = (size_t)n_pages * n_kv * P * HD;
  std::vector<uint16_t> kp(pool_elems, 0x7fc0), vp(pool_elems, 0x7fc0);   // NaN fill: slots past ctx must never be read into the result
  for (int t = 0; t < ctx_len; ++t)
    for (int g = 0; g < n_kv; ++g) {
      const size_t dst = (((size_t)bt[t / P] * n_kv + g) * P + t % P) * HD;
      memcpy(&kp[dst], k_cache + ((size_t)t * n_kv + g) * HD, (size_t)HD * 2);
      memcpy(&vp[dst], v_cache + ((size_t)t * n_kv + g) * HD, (size_t)HD * 2);
    }
  const int qd = n_heads * HD;
  const int pos = ctx_len - 1;
  const int nsplit = std::max(1, std::min(64, sm_count() / n_kv));
  DevBuf dq, dk, dv, dbt, dpos, dout, dpart, dcnt;
  CL_CUDA_OK(dq.upload(q, (size_t)qd * 4));
  CL_CUDA_OK(dk.upload(kp.data(), pool_elems * 2));
  CL_CUDA_OK(dv.upload(vp.data(), pool_elems * 2));
  CL_CUDA_OK(dbt.upload(bt.data(), bt.size() * 4));
  CL_CUDA_OK(dpos.upload(&pos, 4));
  CL_CUDA_OK(dout.alloc((size_t)qd * 4));
  CL_CUDA_OK(dpart.alloc((size_t)n_kv * nsplit * rep * (HD + 2) * 4));
  CL_CUDA_OK(dcnt.alloc((size_t)n_kv * 4));
  CL_CUDA_OK(cudaMemset(dcnt.p, 0, (size_t)n_kv * 4));
  AttnDecodeArgs a;
  a.q = dq.as<float>(); a.q_stride = qd;
  a.kpool = dk.as<__nv_bfloat16>(); a.vpool = dv.as<__nv_bfloat16>(); a.block_tables = dbt.as<int>(); a.bt_stride = n_pages;
  a.pos = dpos.as<int>(); a.out = dout.as<float>(); a.out_stride = qd; a.part = dpart.as<float>(); a.counters = dcnt.as<unsigned>();
  a.batch = 1; a.n_heads = n_heads; a.n_kv = n_kv; a.head_dim = HD; a.page_size = P; a.nsplit = nsplit;
  // run twice: the second launch checks that the split counters re-arm (graph replay safety)
  for (int i = 0; i < 2; ++i)
    if (launch_attn_decode(a, nullptr, false) < 0) { CL_CUDA_OK(cudaGetLastError()); set_last_error("launch_attn_decode failed"); return CL_ERR_CUDA; }
  CL_CUDA_OK(cudaDeviceSynchronize());
  CL_CUDA_OK(cudaMemcpy(out, dout.p, (size_t)qd * 4, cudaMemcpyDeviceToHost));
  return CL_OK;
}

int cl_op_qkv_rope_append(int device, int variant, const uint16_t* w_qkv, const float* h, const float* gain, float eps, int32_t d_model,
                          int32_t n_heads, int32_t n_kv, int32_t head_dim, int32_t pos, float rope_theta, float* q_out,
                          uint16_t* k_out, uint16_t* v_out) {
  if (!w_qkv || !h || !gain || !q_out || !k_out || !v_out || pos < 0) return CL_ERR_INVALID_ARG;
  int rc = check_device(device);
  if (rc) return rc;
  const int HD = head_dim, half = HD / 2, P = 32;
  const int qd = n_heads * HD, kvd = n_kv * HD, rows = qd + 2 * kvd;
  if (!gemv_variant_supported(variant, rows, d_model) || (HD != 64 && HD != 128)) { set_last_error("unsupported shape"); return CL_ERR_INVALID_ARG; }
  // the engine stores q|k|v rows rope-pair-interleaved per head
  std::vector<uint16_t> wp((size_t)rows * d_model);
  for (int r = 0; r < rows; ++r) {
    const int head = r / HD, w = r % HD;
    const int rr = head * HD + (w < half ? 2 * w : 2 * (w - half) + 1);
    memcpy(&wp[(size_t)rr * d_model], w_qkv + (size_t)r * d_model, (size_t)d_model * 2);
  }
  std::vector<float2> rope((size_t)(pos + 1) * half);
  for (int p = 0; p <= pos; ++p)
    for (int i = 0; i < half; ++i) {
      const double inv = pow((double)rope_theta, -2.0 * (double)i / (double)HD);
      rope[(size_t)p * half + i] = make_float2((float)cos((double)p * inv), (float)sin((double)p * inv));
    }
  const int n_pages = pos / P + 1;
  std::vector<int> bt(n_pages);
  for (int i = 0; i < n_pages; ++i) bt[i] = n_pages - 1 - i;
  const size_t pool_elems = (size_t)n_pages * n_kv * P * HD;
  DevBuf dw, dh, dg, dr, dbt, dpos, dq, dk, dv;
  CL_CUDA_OK(dw.upload(wp.data(), wp.size() * 2));
  CL_CUDA_OK(dh.upload(h, (size_t)d_model * 4));
  CL_CUDA_OK(dg.upload(gain, (size_t)d_model * 4));
  CL_CUDA_OK(dr.upload(rope.data(), rope.size() * sizeof(float2)));
  CL_CUDA_OK(dbt.upload(bt.data(), bt.size() * 4));
  CL_CUDA_OK(dpos.upload(&pos, 4));
  CL_CUDA_OK(dq.alloc((size_t)qd * 4));
  CL_CUDA_OK(dk.alloc(pool_elems * 2));
  CL_CUDA_OK(dv.alloc(pool_elems * 2));
  GemvArgs a;
  a.W = dw.as<__nv_bfloat16>(); a.N = rows; a.K = d_model; a.h = dh.as<float>(); a.gain = dg.as<float>(); a.eps = eps;
  a.y = dq.as<float>(); a.x_stride = d_model; a.y_stride = qd; a.batch = 1;
  a.qkv.rope = dr.as<float2>(); a.qkv.pos = dpos.as<int>(); a.qkv.block_tables = dbt.as<int>(); a.qkv.bt_stride = n_pages;
  a.qkv.kpool = dk.as<__nv_bfloat16>(); a.qkv.vpool = dv.as<__nv_bfloat16>();
  a.qkv.n_heads = n_heads; a.qkv.n_kv = n_kv; a.qkv.head_dim = HD; a.qkv.page_size = P;
  if (launch_gemv(variant, EPI_QKV, true, a, nullptr, false) < 0) { CL_CUDA_OK(cudaGetLastError()); return CL_ERR_CUDA; }
  CL_CUDA_OK(cudaDeviceSynchronize());
  CL_CUDA_OK(cudaMemcpy(q_out, dq.p, (size_t)qd * 4, cudaMemcpyDeviceToHost));
  const int page = bt[pos / P], off = pos % P;
  for (int g = 0; g < n_kv; ++g) {
    const size_t src = (((size_t)page * n_kv + g) * P + off) * HD;
    CL_CUDA_OK(cudaMemcpy(k_out + (size_t)g * HD, dk.as<uint16_t>() + src, (size_t)HD * 2, cudaMemcpyDeviceToHost));
    CL_CUDA_OK(cudaMemcpy(v_out + (size_t)g * HD, dv.as<uint16_t>() + src, (size_t)HD * 2, cudaMemcpyDeviceToHost));
  }
  return CL_OK;
}

int cl_op_sample(int device, const float* logits, int32_t n_rows, int32_t vocab, const cl_sampling* s, const int32_t* windows,
                 const int32_t* n_window, const uint64_t* steps, int32_t* ids_out, int32_t iters, float* ms) {
  if (!logits || !s || !windows || !n_window || !steps || !ids_out || n_rows <= 0 || vocab <= 0) return CL_ERR_INVALID_ARG;
  int rc = check_device(device);
  if (rc) return rc;
  const int nblk = sample_blocks(vocab);
  if (!nblk) { set_last_error("vocabulary too large for the device sampler"); return CL_ERR_INVALID_ARG; }
  std::vector<SampleSlot> state((size_t)n_rows);
  for (int r = 0; r < n_rows; ++r) {
    const cl_sampling& sp = s[r];
    const int nw = n_window[r];
    if (!Engine::sample_qualifies(sp, vocab) || nw < 0 || nw > CL_SAMPLE_MAX_WINDOW) {
      set_last_error("row " + std::to_string(r) + ": outside the device sampler's limits");
      return CL_ERR_INVALID_ARG;
    }
    state[r] = Engine::sample_slot(sp, vocab, windows + (size_t)r * CL_SAMPLE_MAX_WINDOW, nw, steps[r]);
  }
  const size_t row_bytes = (size_t)vocab * 4, bytes = (size_t)n_rows * row_bytes;
  DevBuf dl, dst, dpart, dcnt, dtok;
  CL_CUDA_OK(dl.upload(logits, bytes));
  CL_CUDA_OK(dst.upload(state.data(), state.size() * sizeof(SampleSlot)));
  CL_CUDA_OK(dpart.alloc((size_t)n_rows * nblk * kSampleCand * sizeof(unsigned long long)));
  CL_CUDA_OK(dcnt.alloc((size_t)n_rows * 4));
  CL_CUDA_OK(cudaMemset(dcnt.p, 0, (size_t)n_rows * 4));
  CL_CUDA_OK(dtok.alloc((size_t)n_rows * 4));
  SampleArgs a;
  a.logits = dl.as<float>(); a.vocab = vocab; a.state = dst.as<SampleSlot>(); a.tok = dtok.as<int>();
  a.part = dpart.as<unsigned long long>(); a.counters = dcnt.as<unsigned>(); a.batch = n_rows; a.nblk = nblk;
  if (launch_sample(a, nullptr) < 0) { set_last_error(std::string("launch_sample: ") + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; }
  CL_CUDA_OK(cudaDeviceSynchronize());
  CL_CUDA_OK(cudaMemcpy(ids_out, dtok.p, (size_t)n_rows * 4, cudaMemcpyDeviceToHost));
  if (iters > 0 && ms) {
    // timing loop over enough copies of the logits to exceed the 126 MB L2 (each launch reads rows no earlier launch left there)
    const int copies = (int)std::min<size_t>(16, (256ull << 20) / bytes + 1);
    std::vector<DevBuf> extra(copies > 1 ? copies - 1 : 0);
    std::vector<const float*> ls{dl.as<float>()};
    for (auto& b : extra) {
      CL_CUDA_OK(b.alloc(bytes));
      CL_CUDA_OK(cudaMemcpy(b.p, dl.p, bytes, cudaMemcpyDeviceToDevice));
      ls.push_back(b.as<float>());
    }
    cudaEvent_t e0, e1;
    CL_CUDA_OK(cudaEventCreate(&e0));
    CL_CUDA_OK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) { a.logits = ls[i % ls.size()]; launch_sample(a, nullptr); }
    CL_CUDA_OK(cudaDeviceSynchronize());
    CL_CUDA_OK(cudaEventRecord(e0, nullptr));
    for (int i = 0; i < iters; ++i) { a.logits = ls[i % ls.size()]; launch_sample(a, nullptr); }
    CL_CUDA_OK(cudaEventRecord(e1, nullptr));
    CL_CUDA_OK(cudaDeviceSynchronize());
    float t = 0.f;
    CL_CUDA_OK(cudaEventElapsedTime(&t, e0, e1));
    *ms = t / (float)iters;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
  }
  return CL_OK;
}

int cl_op_logprobs(int device, const float* logits, int32_t n_rows, int32_t vocab, const int32_t* chosen, int32_t top_n,
                   float* logprob, int32_t* top_ids, float* top_logprobs, int32_t iters, float* ms) {
  if (!logits || !chosen || !logprob || n_rows <= 0 || vocab <= 0 || top_n < 0 || top_n > CL_MAX_TOP_LOGPROBS ||
      (top_n > 0 && (!top_ids || !top_logprobs)))
    return CL_ERR_INVALID_ARG;
  int rc = check_device(device);
  if (rc) return rc;
  const int nblk = logprob_blocks(vocab);
  if (!nblk) { set_last_error("vocabulary too large for logprobs_kernel"); return CL_ERR_INVALID_ARG; }
  const size_t row_bytes = (size_t)vocab * 4, bytes = (size_t)n_rows * row_bytes;
  DevBuf dl, dtok, drec, dpart, dstat, dcnt;
  CL_CUDA_OK(dl.upload(logits, bytes));
  CL_CUDA_OK(dtok.upload(chosen, (size_t)n_rows * 4));
  CL_CUDA_OK(drec.alloc((size_t)n_rows * sizeof(LogprobRecord)));
  CL_CUDA_OK(dpart.alloc((size_t)n_rows * nblk * CL_MAX_TOP_LOGPROBS * sizeof(unsigned long long)));
  CL_CUDA_OK(dstat.alloc((size_t)n_rows * nblk * sizeof(float2)));
  CL_CUDA_OK(dcnt.alloc((size_t)n_rows * 4));
  CL_CUDA_OK(cudaMemset(dcnt.p, 0, (size_t)n_rows * 4));
  LogprobArgs a;
  a.logits = dl.as<float>(); a.vocab = vocab; a.tok = dtok.as<int>(); a.rec = drec.as<LogprobRecord>();
  a.part = dpart.as<unsigned long long>(); a.stat = dstat.as<float2>(); a.counters = dcnt.as<unsigned>();
  a.batch = n_rows; a.nblk = nblk; a.top_n = top_n;
  if (launch_logprobs(a, nullptr) < 0) { set_last_error(std::string("launch_logprobs: ") + cudaGetErrorString(cudaGetLastError())); return CL_ERR_CUDA; }
  CL_CUDA_OK(cudaDeviceSynchronize());
  std::vector<LogprobRecord> rec((size_t)n_rows);
  CL_CUDA_OK(cudaMemcpy(rec.data(), drec.p, rec.size() * sizeof(LogprobRecord), cudaMemcpyDeviceToHost));
  for (int r = 0; r < n_rows; ++r) {
    logprob[r] = rec[r].logprob;
    for (int j = 0; j < top_n; ++j) {
      top_ids[(size_t)r * top_n + j] = rec[r].top_ids[j];
      top_logprobs[(size_t)r * top_n + j] = rec[r].top_logprobs[j];
    }
  }
  if (iters > 0 && ms) {
    // timing loop over enough copies of the logits to exceed the 126 MB L2 (each launch reads rows no earlier launch left there)
    const int copies = (int)std::min<size_t>(16, (256ull << 20) / bytes + 1);
    std::vector<DevBuf> extra(copies > 1 ? copies - 1 : 0);
    std::vector<const float*> ls{dl.as<float>()};
    for (auto& b : extra) {
      CL_CUDA_OK(b.alloc(bytes));
      CL_CUDA_OK(cudaMemcpy(b.p, dl.p, bytes, cudaMemcpyDeviceToDevice));
      ls.push_back(b.as<float>());
    }
    cudaEvent_t e0, e1;
    CL_CUDA_OK(cudaEventCreate(&e0));
    CL_CUDA_OK(cudaEventCreate(&e1));
    for (int i = 0; i < 3; ++i) { a.logits = ls[i % ls.size()]; launch_logprobs(a, nullptr); }
    CL_CUDA_OK(cudaDeviceSynchronize());
    CL_CUDA_OK(cudaEventRecord(e0, nullptr));
    for (int i = 0; i < iters; ++i) { a.logits = ls[i % ls.size()]; launch_logprobs(a, nullptr); }
    CL_CUDA_OK(cudaEventRecord(e1, nullptr));
    CL_CUDA_OK(cudaDeviceSynchronize());
    float t = 0.f;
    CL_CUDA_OK(cudaEventElapsedTime(&t, e0, e1));
    *ms = t / (float)iters;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
  }
  return CL_OK;
}

int cl_op_synth_weights(int device, uint64_t seed, int32_t tensor_key, int64_t n, float scale, uint16_t* out_bf16) {
  if (!out_bf16 || n <= 0) return CL_ERR_INVALID_ARG;
  int rc = check_device(device);
  if (rc) return rc;
  DevBuf d;
  CL_CUDA_OK(d.alloc((size_t)n * 2));
  if (launch_synth_bf16(d.as<__nv_bfloat16>(), n, (int)std::min<int64_t>(n, 4096), 1, 0, seed, tensor_key, scale, nullptr) < 0) return CL_ERR_CUDA;
  CL_CUDA_OK(cudaDeviceSynchronize());
  CL_CUDA_OK(cudaMemcpy(out_bf16, d.p, (size_t)n * 2, cudaMemcpyDeviceToHost));
  return CL_OK;
}

}  // extern "C"
