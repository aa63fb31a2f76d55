// scheduler.cpp — request-level path: continuous-batching scheduler behind cl_generate().
//
// Replaces what the reference gets from the Ollama server's own scheduler (UPSTREAM of
// /root/reference/pkg/crowdllama/api.go:129-139).  Callers are the per-stream goroutines of
// Peer.handleInferenceRequest (/root/reference/pkg/peer/peer.go:190-256): many may block in
// cl_generate at once; the scheduler thread batches their decode steps (iteration-level
// scheduling) and preempts-by-recompute when the paged KV pool runs dry.
#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>

#include "engine.h"

namespace cl {

static int64_t now_ns() {
  return std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

struct Request {
  std::vector<int32_t> prompt;
  cl_sampling sp{};
  std::vector<int32_t> out;
  cl_seq_t seq = -1;
  int max_new = 0;
  int n_preempted = 0;
  int status = CL_OK;
  std::string done_reason, err;
  bool done = false;
  std::mutex m;
  std::condition_variable cv;
  // streaming: ids the scheduler has published to the waiting client thread (guarded by m); `out` itself is only
  // read by the client after `done`
  bool streaming = false;
  std::vector<int32_t> pub;
  std::vector<LogprobRecord> pub_lp;  // records of `pub` (logprobs requests)
  std::atomic<bool> cancel{false};
  int64_t t_arrive = 0, prefill_ns = 0, decode_ns = 0, t_done = 0;
  uint64_t arrival = 0;
  std::vector<int32_t> full;        // prompt + tokens generated before a preemption: what the (re-)prefill has to process
  size_t prefilled = 0;             // tokens of `full` already in the cache (chunked admission)
  bool dev_sample = false;          // sampled on the device (Engine::sample_qualifies and CL_SCHED_DEVICE_SAMPLE), set at admission
  int top_n = -1;                   // >= 0: log-probabilities asked for, with top_n alternatives
  std::vector<LogprobRecord> lp;    // one record per id of `out` (kept across a preemption, like `out`)
  bool greedy() const { return sp.temperature <= 0.f; }
  bool logprobs() const { return top_n >= 0; }
};

static void fill_result(const Request& r, cl_result* out, const Tokenizer* tok) {
  memset(out, 0, sizeof *out);
  out->n_prompt = (int32_t)r.prompt.size();
  out->n_generated = (int32_t)r.out.size();
  out->token_ids = (int32_t*)malloc(sizeof(int32_t) * std::max<size_t>(1, r.out.size()));
  if (!r.out.empty()) memcpy(out->token_ids, r.out.data(), r.out.size() * 4);
  std::string text = tok ? tok->decode(r.out) : std::string();
  out->text = (char*)malloc(text.size() + 1);
  memcpy(out->text, text.c_str(), text.size() + 1);
  out->text_len = text.size();
  out->done_reason = strdup(r.done_reason.c_str());
  out->prefill_ns = r.prefill_ns;
  out->decode_ns = r.decode_ns;
  out->total_ns = r.t_done - r.t_arrive;
  out->n_preempted = r.n_preempted;
}

static void fill_logprobs(const Request& r, cl_logprobs* out) {
  memset(out, 0, sizeof *out);
  const size_t n = r.lp.size(), k = (size_t)std::max(r.top_n, 0);
  out->n_tokens = (int32_t)n;
  out->top_n = (int32_t)k;
  out->logprob = (float*)malloc(sizeof(float) * std::max<size_t>(1, n));
  if (k) {
    out->top_ids = (int32_t*)malloc(sizeof(int32_t) * std::max<size_t>(1, n * k));
    out->top_logprobs = (float*)malloc(sizeof(float) * std::max<size_t>(1, n * k));
  }
  for (size_t i = 0; i < n; ++i) {
    out->logprob[i] = r.lp[i].logprob;
    for (size_t j = 0; j < k; ++j) {
      out->top_ids[i * k + j] = r.lp[i].top_ids[j];
      out->top_logprobs[i * k + j] = r.lp[i].top_logprobs[j];
    }
  }
}

static void publish(Request& r, int32_t id) {
  if (!r.streaming) return;
  std::lock_guard<std::mutex> lk(r.m);
  r.pub.push_back(id);
  if (r.logprobs()) r.pub_lp.push_back(r.lp.back());
  r.cv.notify_all();
}

// one generated token: `out`, its record (logprobs requests) and the stream.  `row` (host logits the id was drawn from,
// may be nullptr): the record's logprob is taken for that id — the kernel saw the step's argmax in d_tok_.
static void emit_token(Request& r, int32_t id, const LogprobRecord* rec, const float* row) {
  r.out.push_back(id);
  if (r.logprobs()) {
    r.lp.push_back(*rec);
    if (row) r.lp.back().logprob = row[id] - rec->lse;
  }
  publish(r, id);
}

static bool finished(Request& r, const Tokenizer& tok, int max_seq_len) {
  if (r.cancel.load(std::memory_order_relaxed)) { r.done_reason = "cancelled"; return true; }
  if (!r.out.empty() && !r.sp.ignore_eos && tok.is_stop(r.out.back())) { r.done_reason = "stop"; return true; }
  if ((int)r.out.size() >= r.max_new) { r.done_reason = "length"; return true; }
  if ((int)(r.prompt.size() + r.out.size()) >= max_seq_len) { r.done_reason = "length"; return true; }
  return false;
}

// ---- synchronous path (no scheduler thread): one request at a time under the engine lock --------
static int generate_sync(Engine& e, Request& r, const Engine::TokenSink* sink) {
  size_t emitted = 0;
  auto emit = [&]() {
    if (!sink || !sink->fn || r.out.size() <= emitted) return;
    if (sink->fn(sink->user, r.out.data() + emitted, r.logprobs() ? r.lp.data() + emitted : nullptr, (int)(r.out.size() - emitted)))
      r.cancel = true;
    emitted = r.out.size();
  };
  std::lock_guard<std::mutex> lk(e.mu_);
  const int V = e.cfg.vocab_size;
  int rc = e.seq_create(&r.seq);
  if (rc) return rc;
  // a sampled request within the device sampler's limits never copies logits to the host
  r.dev_sample = e.device_sample_ && !r.greedy() && Engine::sample_qualifies(r.sp, V);
  std::vector<float> logits(V);
  int64_t t0 = now_ns();
  rc = e.prefill(r.seq, r.prompt.data(), (int)r.prompt.size(), r.dev_sample ? nullptr : logits.data());
  r.prefill_ns = now_ns() - t0;
  if (rc) { e.seq_free(r.seq); return rc; }
  t0 = now_ns();
  std::vector<int32_t> hist(r.prompt);
  int32_t next = 0;
  LogprobRecord rec;
  if (r.dev_sample) {
    rc = e.sample_setup(r.seq, r.sp, r.prompt.data(), (int)r.prompt.size(), 0);
    if (rc == CL_OK) rc = e.sample_slots(&r.seq, 1, &next);
    if (rc) { e.seq_free(r.seq); return rc; }
  } else {
    next = sample_token(logits.data(), V, r.sp, hist.data(), (int)hist.size(), 0);
  }
  if (r.logprobs() && (rc = e.logprobs_read(&r.seq, 1, r.top_n, &rec)) != CL_OK) { e.seq_free(r.seq); return rc; }
  emit_token(r, next, &rec, r.dev_sample ? nullptr : logits.data());
  emit();
  std::vector<LogprobRecord> recs;
  while (!finished(r, *e.tok, e.cfg.max_seq_len)) {
    if (r.greedy() || r.dev_sample) {
      int room = std::min(r.max_new - (int)r.out.size(), e.cfg.max_seq_len - (int)(r.prompt.size() + r.out.size()));
      int chunk = std::min(room, sink ? 8 : 32);
      std::vector<int32_t> ids(chunk);
      recs.resize(r.logprobs() ? chunk : 0);
      LogprobRecord* lp_out = r.logprobs() ? recs.data() : nullptr;
      const uint64_t step = (uint64_t)r.out.size();
      rc = r.greedy() ? e.decode_greedy(&r.seq, 1, &next, chunk, ids.data(), nullptr, &r.top_n, lp_out)
                      : e.decode_sample(&r.seq, 1, &next, &r.sp, &step, chunk, ids.data(), nullptr, &r.top_n, lp_out);
      if (rc) break;
      for (int i = 0; i < chunk; ++i) {
        emit_token(r, ids[i], lp_out + i, nullptr);
        if (finished(r, *e.tok, e.cfg.max_seq_len)) break;
      }
      next = r.out.back();
    } else {
      rc = e.decode_step(r.seq, next, logits.data(), nullptr);
      if (rc == CL_OK && r.logprobs()) rc = e.logprobs_read(&r.seq, 1, r.top_n, &rec);
      if (rc) break;
      hist.push_back(next);
      next = sample_token(logits.data(), V, r.sp, hist.data(), (int)hist.size(), (uint64_t)r.out.size());
      emit_token(r, next, &rec, logits.data());
    }
    emit();
  }
  r.decode_ns = now_ns() - t0;
  e.seq_free(r.seq);
  r.seq = -1;
  return rc;
}

int Engine::generate_ids(const int32_t* prompt, int n_prompt, const cl_sampling& sp, cl_result* out, const TokenSink* sink,
                         int top_n, cl_logprobs* lp_out) {
  if (!prompt || n_prompt <= 0 || !out) { set_last_error("empty prompt"); return CL_ERR_INVALID_ARG; }
  if (top_n > CL_MAX_TOP_LOGPROBS || (top_n >= 0 && !lp_out)) { set_last_error("top_n outside 0..CL_MAX_TOP_LOGPROBS"); return CL_ERR_INVALID_ARG; }
  if (n_prompt >= cfg.max_seq_len) { set_last_error("prompt longer than max_seq_len"); return CL_ERR_TOO_LONG; }
  for (int i = 0; i < n_prompt; ++i)
    if (prompt[i] < 0 || prompt[i] >= cfg.vocab_size) { set_last_error("token id out of range"); return CL_ERR_INVALID_ARG; }
  auto r = std::make_shared<Request>();
  r->prompt.assign(prompt, prompt + n_prompt);
  r->sp = sp;
  r->max_new = sp.max_new_tokens > 0 ? sp.max_new_tokens : cfg.max_seq_len - n_prompt;
  r->max_new = std::min(r->max_new, cfg.max_seq_len - n_prompt);
  r->t_arrive = now_ns();
  r->streaming = sink && sink->fn;
  r->top_n = top_n < 0 ? -1 : top_n;
  if (!sched_started_) {
    r->status = generate_sync(*this, *r, sink);
    if (r->status == CL_OK) { requests_completed_++; tokens_generated_ += (int64_t)r->out.size(); }
  } else {
    {
      std::lock_guard<std::mutex> lk(q_mu_);
      if (stop_) { set_last_error("engine shutting down"); return CL_ERR_SHUTDOWN; }
      static std::atomic<uint64_t> counter{0};
      r->arrival = counter++;
      queue_.push_back(r);
    }
    q_cv_.notify_all();
    std::unique_lock<std::mutex> lk(r->m);
    size_t seen = 0;
    std::vector<int32_t> fresh;
    std::vector<LogprobRecord> fresh_lp;
    while (true) {
      r->cv.wait(lk, [&] { return r->done || r->pub.size() > seen; });
      if (r->pub.size() > seen) {
        fresh.assign(r->pub.begin() + seen, r->pub.end());
        if (r->logprobs()) fresh_lp.assign(r->pub_lp.begin() + seen, r->pub_lp.end());
        seen = r->pub.size();
        lk.unlock();                       // the callback runs on this (the caller's) thread, outside every lock
        if (sink->fn(sink->user, fresh.data(), r->logprobs() ? fresh_lp.data() : nullptr, (int)fresh.size())) r->cancel = true;
        lk.lock();
        continue;
      }
      if (r->done) break;
    }
  }
  r->t_done = now_ns();
  if (r->status != CL_OK) {
    if (!r->err.empty()) set_last_error(r->err);
    return r->status;
  }
  fill_result(*r, out, tok.get());
  if (r->logprobs()) fill_logprobs(*r, lp_out);
  return CL_OK;
}

void Engine::start_scheduler() {
  if (sched_started_) return;
  stop_ = false;
  sched_started_ = true;
  sched_thread_ = std::thread([this] { scheduler_main(); });
}

void Engine::stop_scheduler() {
  if (!sched_started_) return;
  {
    std::lock_guard<std::mutex> lk(q_mu_);
    stop_ = true;
  }
  q_cv_.notify_all();
  if (sched_thread_.joinable()) sched_thread_.join();
  sched_started_ = false;
}

static void complete(std::shared_ptr<Request>& r, int status, const std::string& err) {
  std::lock_guard<std::mutex> lk(r->m);
  r->status = status;
  r->err = err;
  r->done = true;
  r->cv.notify_all();
}

void Engine::scheduler_main() {
  cudaSetDevice(device_);
  const int V = cfg.vocab_size;
  std::vector<float> logits(V);
  std::vector<int32_t> toks(max_seqs_);
  std::vector<int> slots;
  std::vector<int> last_slots;
  std::vector<cl_seq_t> lp_slots;
  {
    std::lock_guard<std::mutex> elk(mu_);
    {
      const char* v = getenv("CL_SCHED_BLOCKING_SYNC");
      sched_blocking_sync_ = !v || atoi(v) != 0;
      v = getenv("CL_SCHED_MULTI_PREFILL");
      sched_multi_prefill_ = v ? atoi(v) != 0 : kDefaultSchedMultiPrefill != 0;
      v = getenv("CL_SCHED_LINGER_US");
      sched_linger_us_ = v ? atoi(v) : kDefaultSchedLingerUs;
    }
    if (sched_blocking_sync_ && !step_done_ev_ && cudaEventCreateWithFlags(&step_done_ev_, cudaEventBlockingSync | cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError();
      step_done_ev_ = nullptr;
    }
    precapture_graphs();   // every batch size's step graph up front, not inside the first steps that meet it
  }
  while (true) {
    {
      std::unique_lock<std::mutex> lk(q_mu_);
      q_cv_.wait(lk, [&] { return stop_ || !queue_.empty() || !active_.empty() || prefilling_; });
      if (stop_) break;
      // Burst detection while nothing is running: requests of one wave reach the worker over a few milliseconds (one
      // stream per request, pkg/peer/peer.go:177-182).  Waiting as long as new ones keep arriving within
      // sched_linger_us_ of each other (at most 8x that in total) lets the group admission below take them in one
      // pass instead of prefilling the first one alone; a lone request pays sched_linger_us_ once, against a
      // prefill of several milliseconds.
      if (sched_multi_prefill_ && sched_linger_us_ > 0 && active_.empty() && !prefilling_ && !queue_.empty()) {
        const auto t_end = std::chrono::steady_clock::now() + std::chrono::microseconds(8 * (int64_t)sched_linger_us_);
        while ((int)queue_.size() < max_batch_ && std::chrono::steady_clock::now() < t_end) {
          const size_t n = queue_.size();
          if (!q_cv_.wait_for(lk, std::chrono::microseconds(sched_linger_us_), [&] { return stop_ || queue_.size() != n; })) break;   // quiet: go
          if (stop_) break;
        }
        if (stop_) break;
      }
    }
    std::lock_guard<std::mutex> elk(mu_);
    // ---- admission.  A prompt is prefilled in chunks of sched_prefill_chunk_ tokens, ONE chunk per scheduler iteration,
    // interleaved with the decode steps of the running batch: an admit never stalls active sequences for more than one
    // chunk (a 4096-token prompt used to hold every running request for the whole ~85 ms prefill).
    // Several short prompts may be admitted in one iteration as long as their tokens fit the same budget (a burst of
    // 128-token chats fills the batch in a few iterations instead of one request per decode step).
    int budget = sched_prefill_chunk_ > 0 ? sched_prefill_chunk_ : (1 << 30);   // 0: unlimited = whole prompts, as in round 1
    // ---- group admission: the prompts at the head of the queue that fit one pass go through the tile path TOGETHER
    // (Engine::prefill_multi: one weight stream for all of them).  FIFO: the group is a prefix of the queue.  With running
    // sequences the pass is bounded by the same token budget as a chunk; with none to stall, by the workspace (4096 rows).
    if (sched_multi_prefill_ && !prefilling_ && (int)active_.size() < max_batch_ && bws_ && prefill_path_ok()) {
      const int pass_rows = std::min(prefill_chunk_tokens_, prompt_cap_);   // what one prefill_multi pass holds
      const int cap_tokens = active_.empty() ? pass_rows : std::min(budget, pass_rows);
      std::vector<std::shared_ptr<Request>> group;
      {
        std::lock_guard<std::mutex> lk(q_mu_);
        int tokens = 0, pages = 0;
        for (auto& r : queue_) {
          if ((int)(active_.size() + group.size()) >= max_batch_) break;
          const int n = (int)(r->prompt.size() + r->out.size());
          const int need = (n + 1 + page_size_ - 1) / page_size_;
          if (r->cancel.load(std::memory_order_relaxed) || tokens + n > cap_tokens || pages + need > pool_->free_pages()) break;
          group.push_back(r);
          tokens += n;
          pages += need;
        }
        if (group.size() >= 2) queue_.erase(queue_.begin(), queue_.begin() + (long)group.size());
      }
      if (group.size() >= 2) {
        std::vector<cl_seq_t> ss;
        std::vector<const int32_t*> ptrs;
        std::vector<int> lens;
        int rc = CL_OK, total = 0;
        for (auto& r : group) {
          r->full.assign(r->prompt.begin(), r->prompt.end());
          r->full.insert(r->full.end(), r->out.begin(), r->out.end());
          rc = seq_create(&r->seq);
          if (rc == CL_OK) rc = ensure_capacity(r->seq, (int)r->full.size() + 1);
          if (rc) break;
          ss.push_back(r->seq); ptrs.push_back(r->full.data()); lens.push_back((int)r->full.size());
          total += (int)r->full.size();
        }
        const int64_t t0 = now_ns();
        if (rc == CL_OK) rc = prefill_multi((int)ss.size(), ss.data(), ptrs.data(), lens.data(), nullptr);
        const int64_t pdt = now_ns() - t0;
        if (rc == CL_OK) {
          // first tokens of the device-sampled requests: one sampler launch over the group's logits rows
          std::vector<cl_seq_t> dev;
          for (auto& r : group) {
            r->dev_sample = device_sample_ && !r->greedy() && sample_qualifies(r->sp, V);
            if (!r->dev_sample) continue;
            rc = sample_setup(r->seq, r->sp, r->full.data(), (int)r->full.size(), (uint64_t)r->out.size());
            if (rc) break;
            dev.push_back(r->seq);
          }
          if (rc == CL_OK) rc = sample_slots(dev.data(), (int)dev.size(), nullptr);
        }
        if (rc == CL_OK) {
          // the first tokens' log-probabilities: one launch over the group's rows that asked
          std::vector<cl_seq_t> lps;
          int lp_n = -1;
          for (auto& r : group) if (r->logprobs()) { lps.push_back(r->seq); lp_n = std::max(lp_n, r->top_n); }
          if (!lps.empty()) rc = logprobs_enqueue(lps.data(), (int)lps.size(), lp_n);
        }
        if (rc == CL_OK) {
          cudaMemcpyAsync(toks.data(), d_tok_, (size_t)max_seqs_ * 4, cudaMemcpyDeviceToHost, stream_);
          if (cudaStreamSynchronize(stream_) != cudaSuccess) rc = CL_ERR_CUDA;
        }
        sched_prefill_calls_++; sched_prefill_tokens_ += total; sched_prefill_ns_ += pdt;
        if (rc) {
          const std::string err = get_last_error();
          for (auto& r : group) { if (r->seq >= 0) seq_free(r->seq); r->seq = -1; complete(r, rc, err); }
        } else {
          for (auto& r : group) {
            r->prefill_ns += pdt;
            r->prefilled = r->full.size();
            int32_t next = toks[r->seq];                       // greedy: the device argmax of the pass; device-sampled: the draw
            const bool host = !r->greedy() && !r->dev_sample;
            if (host) {
              read_logits(r->seq, logits.data());
              next = sample_token(logits.data(), V, r->sp, r->full.data(), (int)r->full.size(), (uint64_t)r->out.size());
              cudaMemcpyAsync(d_tok_ + r->seq, &next, 4, cudaMemcpyHostToDevice, stream_);
              cudaStreamSynchronize(stream_);
            }
            emit_token(*r, next, r->logprobs() ? &lp_host(r->seq) : nullptr, host ? logits.data() : nullptr);
            if (finished(*r, *tok, cfg.max_seq_len)) {
              seq_free(r->seq);
              requests_completed_++;
              tokens_generated_ += 1;
              complete(r, CL_OK, "");
            } else {
              active_.push_back(r);
            }
          }
        }
        slots_dirty_ = true;
        budget = 0;                        // this iteration's admission is done: on to the decode step
      }
    }
    while (budget > 0) {
      if (!prefilling_ && (int)active_.size() < max_batch_) {
        std::shared_ptr<Request> r;
        {
          std::lock_guard<std::mutex> lk(q_mu_);
          if (!queue_.empty()) r = queue_.front();
        }
        if (r) {
          r->full.assign(r->prompt.begin(), r->prompt.end());
          r->full.insert(r->full.end(), r->out.begin(), r->out.end());
          const int need_pages = ((int)r->full.size() + 1 + page_size_ - 1) / page_size_;
          if (need_pages > pool_->free_pages()) {
            if (active_.empty()) {
              { std::lock_guard<std::mutex> lk(q_mu_); queue_.pop_front(); }
              complete(r, CL_ERR_OOM, "prompt does not fit in the KV page pool");
              continue;
            }
            // else: wait for running requests to release pages
          } else {
            { std::lock_guard<std::mutex> lk(q_mu_); queue_.pop_front(); }
            int rc = seq_create(&r->seq);
            if (rc == CL_OK) rc = ensure_capacity(r->seq, (int)r->full.size() + 1);   // all pages up front: a later chunk cannot run dry
            if (rc) { if (r->seq >= 0) seq_free(r->seq); r->seq = -1; complete(r, rc, get_last_error()); continue; }
            r->prefilled = 0;
            r->dev_sample = device_sample_ && !r->greedy() && sample_qualifies(r->sp, V);
            prefilling_ = r;
          }
        }
      }
      if (!prefilling_) break;
      auto r = prefilling_;
      if (r->cancel.load(std::memory_order_relaxed)) {
        seq_free(r->seq); r->seq = -1; r->done_reason = "cancelled"; prefilling_.reset();
        requests_completed_++;
        complete(r, CL_OK, "");
        continue;
      }
      const size_t left = r->full.size() - r->prefilled;
      const size_t chunk = active_.empty() ? left : std::min(left, (size_t)budget);   // nobody to stall: the whole prompt at once
      const bool last = chunk == left;
      const int64_t t0 = now_ns();
      int rc = prefill(r->seq, r->full.data() + r->prefilled, (int)chunk, last && !r->dev_sample ? logits.data() : nullptr);
      const int64_t pdt = now_ns() - t0;
      r->prefill_ns += pdt;
      sched_prefill_calls_++; sched_prefill_tokens_ += (int64_t)chunk; sched_prefill_ns_ += pdt;
      slots_dirty_ = true;                // prefill rewrote d_slots_[0]
      budget -= (int)std::min(chunk, (size_t)budget);
      if (rc) { seq_free(r->seq); r->seq = -1; prefilling_.reset(); complete(r, rc, get_last_error()); continue; }
      r->prefilled += chunk;
      if (!last) break;                   // budget used up in the middle of a prompt
      prefilling_.reset();
      int32_t next = 0;
      if (r->dev_sample) {
        rc = sample_setup(r->seq, r->sp, r->full.data(), (int)r->full.size(), (uint64_t)r->out.size());
        if (rc == CL_OK) rc = sample_slots(&r->seq, 1, &next);
        if (rc) { seq_free(r->seq); r->seq = -1; complete(r, rc, get_last_error()); continue; }
      } else {
        next = sample_token(logits.data(), V, r->sp, r->full.data(), (int)r->full.size(), (uint64_t)r->out.size());
      }
      LogprobRecord rec;
      if (r->logprobs() && (rc = logprobs_read(&r->seq, 1, r->top_n, &rec)) != CL_OK) {
        seq_free(r->seq); r->seq = -1; complete(r, rc, get_last_error()); continue;
      }
      emit_token(*r, next, &rec, r->dev_sample ? nullptr : logits.data());
      if (!r->greedy() && !r->dev_sample) cudaMemcpyAsync(d_tok_ + r->seq, &r->out.back(), 4, cudaMemcpyHostToDevice, stream_);
      if (finished(*r, *tok, cfg.max_seq_len)) {
        seq_free(r->seq);
        requests_completed_++;
        tokens_generated_ += 1;
        complete(r, CL_OK, "");
      } else {
        active_.push_back(r);
      }
    }
    if (active_.empty()) continue;
    // ---- make room for one more token per active request; preempt the youngest on OOM
    for (size_t i = 0; i < active_.size();) {
      auto& r = active_[i];
      int rc = ensure_capacity(r->seq, seqs_[r->seq].len + 1);
      if (rc == CL_ERR_OOM && prefilling_) {
        // the request still being admitted is the youngest of all: it gives its pages back and waits at the queue's head
        auto v = prefilling_;
        seq_free(v->seq);
        v->seq = -1;
        v->n_preempted++;
        preemptions_++;
        prefilling_.reset();
        { std::lock_guard<std::mutex> lk(q_mu_); queue_.push_front(v); }
        continue;                       // retry this request's capacity
      }
      if (rc == CL_ERR_OOM && active_.size() > 1) {
        size_t victim = 0;
        for (size_t k = 1; k < active_.size(); ++k) if (active_[k]->arrival > active_[victim]->arrival) victim = k;
        auto v = active_[victim];
        seq_free(v->seq);
        v->seq = -1;
        v->n_preempted++;
        preemptions_++;
        active_.erase(active_.begin() + victim);
        { std::lock_guard<std::mutex> lk(q_mu_); queue_.push_front(v); }
        i = 0;  // restart the capacity pass
        continue;
      }
      if (rc) {
        seq_free(r->seq);
        auto dead = r;
        active_.erase(active_.begin() + i);
        complete(dead, rc, get_last_error());
        continue;
      }
      ++i;
    }
    if (active_.empty()) continue;
    // ---- one batched decode step
    const int B = (int)active_.size();
    slots.resize(B);
    for (int b = 0; b < B; ++b) slots[b] = active_[b]->seq;
    // slots_dirty_: an admission-time prefill (or a token-level call) rewrote d_slots_[0] since the last upload — the
    // cached list would leave a finished request's slot in place and every later step would run on it
    if (slots != last_slots || slots_dirty_) {
      cudaMemcpyAsync(d_slots_, slots.data(), (size_t)B * 4, cudaMemcpyHostToDevice, stream_);
      last_slots = slots;
      slots_dirty_ = false;
      last_single_slot_ = B == 1 ? slots[0] : -1;
    }
    const int64_t t0 = now_ns();
    int rc = run_step_graph(B);
    // the device sampler overwrites the step's argmax of the device-sampled slots (one launch for the whole batch)
    if (rc == CL_OK && std::any_of(active_.begin(), active_.end(), [](const std::shared_ptr<Request>& r) { return r->dev_sample; }))
      rc = launch_sampler(B, d_slots_, false);
    // log-probabilities of the rows that asked (one launch; nothing at all when no row did)
    lp_slots.clear();
    int lp_n = -1;
    for (auto& r : active_) if (r->logprobs()) { lp_slots.push_back(r->seq); lp_n = std::max(lp_n, r->top_n); }
    if (rc == CL_OK && !lp_slots.empty()) rc = logprobs_enqueue(lp_slots.data(), (int)lp_slots.size(), lp_n);
    if (rc == CL_OK) {
      cudaMemcpyAsync(toks.data(), d_tok_, (size_t)max_seqs_ * 4, cudaMemcpyDeviceToHost, stream_);
      // Batched steps last 3.5-6 ms: wait on a blocking-sync event instead of spinning in cudaStreamSynchronize, so that
      // eight worker processes on one box do not burn eight host cores (the box's cgroup quota is 16) while their GPUs
      // work.  Single-sequence steps (2.8 ms, latency matters) keep the spinning wait.
      if (B >= 2 && sched_blocking_sync_ && step_done_ev_) {
        if (cudaEventRecord(step_done_ev_, stream_) != cudaSuccess || cudaEventSynchronize(step_done_ev_) != cudaSuccess) rc = CL_ERR_CUDA;
      } else if (cudaStreamSynchronize(stream_) != cudaSuccess) rc = CL_ERR_CUDA;
    }
    if (rc) {
      const std::string err = get_last_error();
      for (auto& r : active_) { seq_free(r->seq); complete(r, rc, err); }
      active_.clear();
      last_slots.clear();
      continue;
    }
    for (int b = 0; b < B; ++b) {
      auto& r = active_[b];
      auto& st = seqs_[r->seq];
      st.history.push_back(r->out.back());
      st.len += 1;
      int32_t next = toks[r->seq];
      const bool host = !r->greedy() && !r->dev_sample;
      if (host) {
        read_logits(r->seq, logits.data());
        next = sample_token(logits.data(), V, r->sp, st.history.data(), (int)st.history.size(), (uint64_t)r->out.size());
        cudaMemcpyAsync(d_tok_ + r->seq, &next, 4, cudaMemcpyHostToDevice, stream_);
        cudaStreamSynchronize(stream_);
      }
      emit_token(*r, next, r->logprobs() ? &lp_host(r->seq) : nullptr, host ? logits.data() : nullptr);
    }
    const int64_t dt = now_ns() - t0;
    for (auto& r : active_) r->decode_ns += dt;
    tokens_generated_ += B;
    sched_decode_steps_++; sched_decode_ns_ += dt;
    const double tps = (double)max_batch_ / ((double)dt * 1e-9);   // capacity at the current step time (engine.cu, init)
    tok_per_sec_ewma_ = tok_per_sec_ewma_ == 0.0 ? tps : 0.9 * tok_per_sec_ewma_ + 0.1 * tps;
    // ---- retire finished requests
    for (size_t i = 0; i < active_.size();) {
      auto r = active_[i];
      if (finished(*r, *tok, cfg.max_seq_len)) {
        seq_free(r->seq);
        active_.erase(active_.begin() + i);
        requests_completed_++;
        complete(r, CL_OK, "");
      } else {
        ++i;
      }
    }
  }
  // shutdown: fail whatever is left
  std::lock_guard<std::mutex> elk(mu_);
  for (auto& r : active_) { if (r->seq >= 0) seq_free(r->seq); complete(r, CL_ERR_SHUTDOWN, "engine shutting down"); }
  active_.clear();
  if (prefilling_) { if (prefilling_->seq >= 0) seq_free(prefilling_->seq); complete(prefilling_, CL_ERR_SHUTDOWN, "engine shutting down"); prefilling_.reset(); }
  std::deque<std::shared_ptr<Request>> rest;
  { std::lock_guard<std::mutex> lk(q_mu_); rest.swap(queue_); }
  for (auto& r : rest) complete(r, CL_ERR_SHUTDOWN, "engine shutting down");
}

}  // namespace cl
