// capi.cpp — extern "C" entry points declared in include/clengine.h.
#include <chrono>
#include <cstdlib>
#include <cstring>

#include "engine.h"

using namespace cl;

extern "C" {

int cl_abi_version(void) { return CL_ABI_VERSION; }

const char* cl_strerror(int status) {
  switch (status) {
    case CL_OK: return "ok";
    case CL_ERR_INVALID_ARG: return "invalid argument";
    case CL_ERR_NO_DEVICE: return "no sm_100 CUDA device (no CPU fallback)";
    case CL_ERR_CUDA: return "CUDA error";
    case CL_ERR_OOM: return "out of device memory or KV pages";
    case CL_ERR_UNKNOWN_MODEL: return "model not served by this engine";
    case CL_ERR_TOO_LONG: return "sequence exceeds max_seq_len";
    case CL_ERR_BAD_SEQ: return "bad sequence handle";
    case CL_ERR_SHUTDOWN: return "engine shutting down";
    case CL_ERR_IO: return "I/O error";
    case CL_ERR_INTERNAL: return "internal error";
    case CL_ERR_BAD_MESSAGE: return "expected GenerateRequest, got different message type";
    default: return "unknown status";
  }
}

const char* cl_last_error(void) { return get_last_error(); }

void cl_default_engine_config(cl_engine_config* c) {
  memset(c, 0, sizeof *c);
  c->abi_version = CL_ABI_VERSION;
  c->page_size = 32;
  c->max_batch = 8;
  c->max_seqs = 8;
  c->use_cuda_graph = 1;
  c->weights_seed = 1234;
}

void cl_default_sampling(cl_sampling* s) {
  memset(s, 0, sizeof *s);
  s->temperature = 0.8f;
  s->top_k = 40;
  s->top_p = 0.9f;
  s->repeat_penalty = 1.1f;
  s->repeat_last_n = 64;
  s->seed = (uint64_t)std::chrono::steady_clock::now().time_since_epoch().count();
  s->max_new_tokens = -1;
}

int cl_sample_token(const float* logits, int32_t vocab, const cl_sampling* s, const int32_t* history, int32_t n_history,
                    uint64_t step, int32_t* id) {
  if (!logits || vocab <= 0 || !s || !id || n_history < 0 || (n_history > 0 && !history)) return CL_ERR_INVALID_ARG;
  *id = cl::sample_token(logits, vocab, *s, history, n_history, step);
  return CL_OK;
}

void cl_greedy_sampling(cl_sampling* s, int32_t max_new_tokens) {
  memset(s, 0, sizeof *s);
  s->temperature = 0.f;
  s->repeat_penalty = 1.f;
  s->max_new_tokens = max_new_tokens;
}

int cl_model_preset(const char* name, cl_model_config* o) {
  if (!name || !o) return CL_ERR_INVALID_ARG;
  struct P { const char* n; cl_model_config c; };
  static const P presets[] = {
      {"llama3-8b", {32, 4096, 32, 8, 128, 14336, 128256, 8192, 5e5f, 1e-5f}},
      {"mistral-7b", {32, 4096, 32, 8, 128, 14336, 32000, 8192 + 512, 1e6f, 1e-5f}},
      {"tinyllama-1.1b", {22, 2048, 32, 4, 64, 5632, 32000, 2048, 1e4f, 1e-5f}},
      // "llama3" rotary scaling (factor, low / high frequency factor, original context): Llama-3.1 and 3.2
      {"llama3.1-8b", {32, 4096, 32, 8, 128, 14336, 128256, 32768, 5e5f, 1e-5f, 8.f, 1.f, 4.f, 8192}},
      {"llama3.2-1b", {16, 2048, 32, 8, 64, 8192, 128256, 8192, 5e5f, 1e-5f, 32.f, 1.f, 4.f, 8192}},
      {"tiny-test", {2, 256, 4, 2, 64, 512, 512, 512, 1e4f, 1e-5f}},
  };
  for (const auto& p : presets)
    if (!strcmp(p.n, name)) { *o = p.c; return CL_OK; }
  return CL_ERR_UNKNOWN_MODEL;
}

int cl_engine_create(const cl_engine_config* cfg, cl_engine** out) {
  if (!cfg || !out) return CL_ERR_INVALID_ARG;
  *out = nullptr;
  cl_engine* e = new (std::nothrow) cl_engine();
  if (!e) return CL_ERR_OOM;
  int rc;
  try {
    rc = e->impl.init(*cfg);
  } catch (const std::exception& ex) {
    set_last_error(ex.what());
    rc = CL_ERR_INTERNAL;
  }
  if (rc) {
    std::string keep = get_last_error();
    delete e;
    cudaGetLastError();
    set_last_error(keep);
    return rc;
  }
  *out = e;
  return CL_OK;
}

void cl_engine_destroy(cl_engine* e) { delete e; }

int cl_engine_model_config(const cl_engine* e, cl_model_config* out) {
  if (!e || !out) return CL_ERR_INVALID_ARG;
  *out = e->impl.cfg;
  return CL_OK;
}

int cl_engine_stats(cl_engine* e, cl_stats* out) {
  if (!e || !out) return CL_ERR_INVALID_ARG;
  return e->impl.stats(out);
}

int cl_engine_set_tensor(cl_engine* e, int32_t layer, int32_t kind, const uint16_t* data, int64_t n) {
  if (!e || !data) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  return e->impl.set_tensor(layer, kind, data, n);
}

#define CL_GUARD(...)                                   \
  try { __VA_ARGS__ }                                        \
  catch (const std::exception& ex) { set_last_error(ex.what()); return CL_ERR_INTERNAL; }

int cl_generate_ids(cl_engine* e, const int32_t* prompt_ids, int32_t n_prompt, const cl_sampling* s, cl_result* out) {
  if (!e || !out) return CL_ERR_INVALID_ARG;
  cl_sampling sp;
  if (s) sp = *s; else cl_default_sampling(&sp);
  CL_GUARD(return e->impl.generate_ids(prompt_ids, n_prompt, sp, out);)
}

int cl_generate_ids_logprobs(cl_engine* e, const int32_t* prompt_ids, int32_t n_prompt, const cl_sampling* s, int32_t top_n,
                             cl_result* out, cl_logprobs* lp) {
  if (!e || !out || !lp || top_n < 0 || top_n > CL_MAX_TOP_LOGPROBS) return CL_ERR_INVALID_ARG;
  cl_sampling sp;
  if (s) sp = *s; else cl_default_sampling(&sp);
  CL_GUARD(return e->impl.generate_ids(prompt_ids, n_prompt, sp, out, nullptr, top_n, lp);)
}

void cl_logprobs_free(cl_logprobs* l) {
  if (!l) return;
  free(l->logprob);
  free(l->top_ids);
  free(l->top_logprobs);
  memset(l, 0, sizeof *l);
}

namespace {
// incremental detokeniser: emits only text that later tokens cannot change (an incomplete UTF-8 tail is held back)
struct StreamText {
  const Tokenizer* tok;
  std::vector<int32_t> ids;
  size_t emitted = 0;       // bytes of sanitised text already handed out
  std::string feed(const int32_t* fresh, int n, bool final) {
    ids.insert(ids.end(), fresh, fresh + n);
    std::string raw = tok->decode_bytes(ids);
    size_t cut = raw.size();
    if (!final) {
      for (size_t back = 1; back <= 3 && back <= raw.size(); ++back) {
        const unsigned char c = (unsigned char)raw[raw.size() - back];
        if ((c >> 6) == 2) continue;                                   // continuation byte: keep looking for the lead
        const size_t need = (c >> 5) == 6 ? 2 : (c >> 4) == 14 ? 3 : (c >> 3) == 30 ? 4 : 1;
        if (need > back) cut = raw.size() - back;                      // lead byte of a sequence that is still open
        break;
      }
    }
    const std::string stable = Tokenizer::sanitize(raw.substr(0, cut));
    std::string delta = stable.size() > emitted ? stable.substr(emitted) : std::string();
    emitted = std::max(emitted, stable.size());
    return delta;
  }
};
struct TextSinkCtx { StreamText st; cl_token_cb cb; void* user; };
int text_sink(void* u, const int32_t* ids, const LogprobRecord*, int n) {
  auto* c = (TextSinkCtx*)u;
  const std::string delta = c->st.feed(ids, n, false);
  return c->cb(c->user, delta.data(), delta.size(), ids, n);
}
int64_t wall_ns() {
  return std::chrono::duration_cast<std::chrono::nanoseconds>(std::chrono::system_clock::now().time_since_epoch()).count();
}
std::vector<uint8_t> response_frame(const std::string& model, const std::string& text, bool done, const std::string& reason,
                                    std::vector<PbTokenLogprob> logprobs = {}) {
  PbGenerateResponse pr;
  pr.logprobs = std::move(logprobs);
  pr.model = model;
  const int64_t ns = wall_ns();
  pr.created_at_sec = ns / 1000000000ll;
  pr.created_at_nanos = (int32_t)(ns % 1000000000ll);
  pr.response = text;
  pr.done = done;
  pr.done_reason = reason;
  pr.worker_id = "worker";                 // api.go:83 (literal in the reference)
  pr.total_duration = done ? ns : 0;       // api.go:84: the reference stores time.Now().UnixNano() here
  return pb_encode_response(pr);
}
// GenerateResponse.logprobs entry of one generated id
PbTokenLogprob token_logprob(const Tokenizer& tok, int32_t id, const LogprobRecord& r, int top_n) {
  PbTokenLogprob t;
  t.token = tok.token_bytes(id);
  t.logprob = r.logprob;
  for (int j = 0; j < top_n; ++j) {
    if (r.top_ids[j] < 0) break;                     // a vocabulary smaller than top_n
    t.top_logprobs.push_back(PbTopLogprob{tok.token_bytes(r.top_ids[j]), r.top_logprobs[j]});
  }
  return t;
}
// a frame carries the records of the ids its text covers: ids whose bytes are held back (an open UTF-8 sequence) wait
// for the next frame, the final frame takes whatever is left
struct FrameSinkCtx {
  StreamText st; cl_frame_cb cb; void* user; std::string model;
  int top_n = -1;
  std::vector<PbTokenLogprob> pending;
};
int frame_sink(void* u, const int32_t* ids, const LogprobRecord* lp, int n) {
  auto* c = (FrameSinkCtx*)u;
  if (lp && c->top_n >= 0)
    for (int i = 0; i < n; ++i) c->pending.push_back(token_logprob(*c->st.tok, ids[i], lp[i], c->top_n));
  const std::string delta = c->st.feed(ids, n, false);
  if (delta.empty()) return 0;
  const std::vector<uint8_t> f = response_frame(c->model, delta, false, "", std::move(c->pending));
  c->pending.clear();
  return c->cb(c->user, f.data(), f.size());
}
int check_model(cl_engine* e, const char* model) {
  // exact string match, like Resource.SupportedModels (manager.go:349-354)
  if (model && *model && e->impl.model_name != model) {
    set_last_error(std::string("model '") + model + "' is not served (serving '" + e->impl.model_name + "')");
    return CL_ERR_UNKNOWN_MODEL;
  }
  return CL_OK;
}
std::vector<int32_t> prompt_ids(cl_engine* e, const char* prompt, size_t prompt_len, bool raw) {
  const std::string user(prompt, prompt_len);
  return e->impl.tok->encode(raw ? user : e->impl.tok->apply_chat_template(user), true);
}
}  // namespace

int cl_generate(cl_engine* e, const char* model, const char* prompt, size_t prompt_len, const cl_sampling* s, cl_result* out) {
  if (!e || !prompt || !out) return CL_ERR_INVALID_ARG;
  if (int rc = check_model(e, model)) return rc;
  CL_GUARD(
    std::vector<int32_t> ids = prompt_ids(e, prompt, prompt_len, false);
    cl_sampling sp;
    if (s) sp = *s; else cl_default_sampling(&sp);
    return e->impl.generate_ids(ids.data(), (int)ids.size(), sp, out);
  )
}

int cl_generate_stream(cl_engine* e, const char* model, const char* prompt, size_t prompt_len, const cl_sampling* s, cl_token_cb cb,
                       void* user, cl_result* out) {
  if (!e || !prompt || !out || !cb) return CL_ERR_INVALID_ARG;
  if (int rc = check_model(e, model)) return rc;
  CL_GUARD(
    std::vector<int32_t> ids = prompt_ids(e, prompt, prompt_len, false);
    cl_sampling sp;
    if (s) sp = *s; else cl_default_sampling(&sp);
    TextSinkCtx ctx{StreamText{e->impl.tok.get(), {}, 0}, cb, user};
    Engine::TokenSink sink{text_sink, &ctx};
    const int rc = e->impl.generate_ids(ids.data(), (int)ids.size(), sp, out, &sink);
    if (rc) return rc;
    const std::string tail = ctx.st.feed(nullptr, 0, true);   // whatever the UTF-8 hold-back kept
    if (!tail.empty()) cb(user, tail.data(), tail.size(), nullptr, 0);
    return CL_OK;
  )
}

void cl_result_free(cl_result* r) {
  if (!r) return;
  free(r->text);
  free(r->done_reason);
  free(r->token_ids);
  memset(r, 0, sizeof *r);
}

static int handle_message_impl(cl_engine* e, const uint8_t* req, size_t req_len, const cl_sampling* s, cl_frame_cb cb, void* user,
                               bool allow_stream) {
  PbGenerateRequest gr;
  if (!pb_decode_request(req, req_len, &gr)) {
    set_last_error("expected GenerateRequest, got different message type");  // api.go:50
    return CL_ERR_BAD_MESSAGE;
  }
  if (int rc = check_model(e, gr.model.c_str())) return rc;
  cl_sampling sp;
  if (s) sp = *s; else cl_default_sampling(&sp);
  apply_options(gr.opt, &sp);                                   // request options win over the worker's defaults
  // log-probabilities (options fields 9 / 10): top_logprobs alone asks for nothing, as in Ollama
  int top_n = -1;
  if (gr.opt.logprobs) {
    top_n = gr.opt.top_logprobs;
    if (top_n < 0 || top_n > CL_MAX_TOP_LOGPROBS) {
      set_last_error("top_logprobs must be within 0.." + std::to_string(CL_MAX_TOP_LOGPROBS));
      return CL_ERR_INVALID_ARG;
    }
  }
  std::vector<int32_t> ids = prompt_ids(e, gr.prompt.data(), gr.prompt.size(), gr.opt.raw);
  cl_result r;
  cl_logprobs lp{};
  if (gr.stream && allow_stream) {
    // streaming (SURVEY.md §8f row 4): Done=false frames carrying text deltas, then one Done=true frame
    FrameSinkCtx ctx{StreamText{e->impl.tok.get(), {}, 0}, cb, user, gr.model, top_n, {}};
    Engine::TokenSink sink{frame_sink, &ctx};
    const int rc = e->impl.generate_ids(ids.data(), (int)ids.size(), sp, &r, &sink, top_n, &lp);
    if (rc) return rc;
    const std::string tail = ctx.st.feed(nullptr, 0, true);
    const std::vector<uint8_t> f = response_frame(gr.model, tail, true, r.done_reason, std::move(ctx.pending));
    cl_result_free(&r);
    cl_logprobs_free(&lp);
    cb(user, f.data(), f.size());
    return CL_OK;
  }
  const int rc = e->impl.generate_ids(ids.data(), (int)ids.size(), sp, &r, nullptr, top_n, &lp);
  if (rc) return rc;
  std::vector<PbTokenLogprob> entries;
  for (int i = 0; top_n >= 0 && i < lp.n_tokens; ++i) {
    LogprobRecord rec;
    rec.logprob = lp.logprob[i];
    for (int j = 0; j < lp.top_n; ++j) { rec.top_ids[j] = lp.top_ids[i * lp.top_n + j]; rec.top_logprobs[j] = lp.top_logprobs[i * lp.top_n + j]; }
    entries.push_back(token_logprob(*e->impl.tok, r.token_ids[i], rec, lp.top_n));
  }
  const std::vector<uint8_t> f = response_frame(gr.model, std::string(r.text, r.text_len), true, r.done_reason, std::move(entries));
  cl_result_free(&r);
  cl_logprobs_free(&lp);
  cb(user, f.data(), f.size());
  return CL_OK;
}

static int collect_frame(void* user, const uint8_t* msg, size_t len) {
  auto* v = (std::vector<uint8_t>*)user;
  v->assign(msg, msg + len);
  return 0;
}

int cl_handle_message(cl_engine* e, const uint8_t* req, size_t req_len, const cl_sampling* s, uint8_t** resp, size_t* resp_len) {
  if (!e || !req || !resp || !resp_len) return CL_ERR_INVALID_ARG;
  *resp = nullptr;
  *resp_len = 0;
  CL_GUARD(
    std::vector<uint8_t> b;
    const int rc = handle_message_impl(e, req, req_len, s, collect_frame, &b, false);   // one complete answer (api.go:77-92)
    if (rc) return rc;
    *resp = (uint8_t*)malloc(b.size() ? b.size() : 1);
    memcpy(*resp, b.data(), b.size());
    *resp_len = b.size();
    return CL_OK;
  )
}

int cl_handle_message_stream(cl_engine* e, const uint8_t* req, size_t req_len, const cl_sampling* s, cl_frame_cb cb, void* user) {
  if (!e || !req || !cb) return CL_ERR_INVALID_ARG;
  CL_GUARD(return handle_message_impl(e, req, req_len, s, cb, user, true);)
}

void cl_buffer_free(void* p) { free(p); }

// ---- tokenizer (tokenizer.cpp) ---------------------------------------------------------------------------------
struct cl_tokenizer { std::unique_ptr<Tokenizer> t; };

int cl_tokenizer_load(const char* tokenizer_json_path, const char* chat_family, cl_tokenizer** out) {
  if (!tokenizer_json_path || !out) return CL_ERR_INVALID_ARG;
  *out = nullptr;
  CL_GUARD(
    std::string err;
    std::unique_ptr<Tokenizer> t = load_hf_tokenizer(tokenizer_json_path, chat_family ? chat_family : "", &err);
    if (!t) { set_last_error(err); return CL_ERR_IO; }
    *out = new cl_tokenizer{std::move(t)};
    return CL_OK;
  )
}
void cl_tokenizer_free(cl_tokenizer* t) { delete t; }
int cl_tokenizer_encode(const cl_tokenizer* t, const char* text, size_t len, int32_t add_bos, int32_t chat, int32_t* ids, int32_t cap,
                        int32_t* n_out) {
  if (!t || !text || !n_out) return CL_ERR_INVALID_ARG;
  CL_GUARD(
    const std::string s(text, len);
    const std::vector<int32_t> v = t->t->encode(chat ? t->t->apply_chat_template(s) : s, add_bos != 0);
    *n_out = (int32_t)v.size();
    if (ids && cap >= (int32_t)v.size()) { if (!v.empty()) memcpy(ids, v.data(), v.size() * 4); }
    else if (ids) return CL_ERR_INVALID_ARG;
    return CL_OK;
  )
}
int cl_tokenizer_decode(const cl_tokenizer* t, const int32_t* ids, int32_t n, char* buf, size_t cap, size_t* len_out) {
  if (!t || (!ids && n > 0) || !len_out) return CL_ERR_INVALID_ARG;
  CL_GUARD(
    const std::string s = t->t->decode_bytes(std::vector<int32_t>(ids, ids + n));   // raw bytes: the caller decides about UTF-8
    *len_out = s.size();
    if (buf && cap >= s.size()) { if (!s.empty()) memcpy(buf, s.data(), s.size()); }
    else if (buf) return CL_ERR_INVALID_ARG;
    return CL_OK;
  )
}
int cl_tokenizer_info(const cl_tokenizer* t, int32_t* vocab_size, int32_t* bos, int32_t* eos) {
  if (!t) return CL_ERR_INVALID_ARG;
  if (vocab_size) *vocab_size = t->t->vocab_size();
  if (bos) *bos = t->t->bos();
  if (eos) *eos = t->t->eos();
  return CL_OK;
}
int cl_engine_load_tokenizer(cl_engine* e, const char* tokenizer_json_path, const char* chat_family) {
  if (!e || !tokenizer_json_path) return CL_ERR_INVALID_ARG;
  CL_GUARD(
    std::string err;
    std::unique_ptr<Tokenizer> t = load_hf_tokenizer(tokenizer_json_path, chat_family ? chat_family : "", &err);
    if (!t) { set_last_error(err); return CL_ERR_IO; }
    if (t->vocab_size() > e->impl.cfg.vocab_size) {
      set_last_error("tokenizer has more ids than the model's vocabulary");
      return CL_ERR_INVALID_ARG;
    }
    std::lock_guard<std::mutex> lk(e->impl.mu_);
    e->impl.tok = std::move(t);
    return CL_OK;
  )
}

int cl_tokenize(cl_engine* e, const char* text, size_t len, int32_t* ids, int32_t cap, int32_t* n_out) {
  if (!e || !text || !n_out) return CL_ERR_INVALID_ARG;
  std::vector<int32_t> v = e->impl.tok->encode(std::string(text, len), false);
  *n_out = (int32_t)v.size();
  if (ids && cap >= (int32_t)v.size()) memcpy(ids, v.data(), v.size() * 4);
  else if (ids) return CL_ERR_INVALID_ARG;
  return CL_OK;
}

int cl_detokenize(cl_engine* e, const int32_t* ids, int32_t n, char* buf, size_t cap, size_t* len_out) {
  if (!e || !ids || !len_out) return CL_ERR_INVALID_ARG;
  std::string s = e->impl.tok->decode(std::vector<int32_t>(ids, ids + n));
  *len_out = s.size();
  if (buf) {
    if (cap < s.size() + 1) return CL_ERR_INVALID_ARG;
    memcpy(buf, s.c_str(), s.size() + 1);
  }
  return CL_OK;
}

int cl_seq_create(cl_engine* e, cl_seq_t* out) {
  if (!e || !out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  return e->impl.seq_create(out);
}
int cl_seq_free(cl_engine* e, cl_seq_t s) {
  if (!e) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  return e->impl.seq_free(s);
}
int cl_seq_len(cl_engine* e, cl_seq_t s, int32_t* len_out) {
  if (!e || !len_out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  return e->impl.seq_len(s, len_out);
}
int cl_prefill(cl_engine* e, cl_seq_t s, const int32_t* ids, int32_t n, float* logits_out) {
  if (!e || !ids) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.prefill(s, ids, n, logits_out);)
}
int cl_prefill_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs, const int32_t* ids, const int32_t* lens, float* logits_out) {
  if (!e || !seqs || !ids || !lens || n_seqs <= 0) return CL_ERR_INVALID_ARG;
  std::vector<const int32_t*> ptrs((size_t)n_seqs);
  size_t off = 0;
  for (int i = 0; i < n_seqs; ++i) {
    if (lens[i] <= 0) return CL_ERR_INVALID_ARG;
    ptrs[(size_t)i] = ids + off;
    off += (size_t)lens[i];
  }
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.prefill_multi(n_seqs, seqs, ptrs.data(), lens, logits_out);)
}
int cl_decode_step(cl_engine* e, cl_seq_t s, int32_t id, float* logits_out, int32_t* argmax_out) {
  if (!e) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.decode_step(s, id, logits_out, argmax_out);)
}
int cl_decode_greedy(cl_engine* e, cl_seq_t s, int32_t first_id, int32_t n_steps, int32_t* ids_out, float* device_ms) {
  if (!e || !ids_out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.decode_greedy(&s, 1, &first_id, n_steps, ids_out, device_ms);)
}
int cl_decode_greedy_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs, const int32_t* first_ids, int32_t n_steps,
                           int32_t* ids_out, float* device_ms) {
  if (!e || !seqs || !first_ids || !ids_out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.decode_greedy(seqs, n_seqs, first_ids, n_steps, ids_out, device_ms);)
}
int cl_decode_sample_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs, const int32_t* first_ids, const cl_sampling* s,
                           const uint64_t* first_steps, int32_t n_steps, int32_t* ids_out, float* device_ms) {
  if (!e || !seqs || !first_ids || !s || !first_steps || !ids_out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.decode_sample(seqs, n_seqs, first_ids, s, first_steps, n_steps, ids_out, device_ms);)
}
int cl_decode_step_batch(cl_engine* e, const cl_seq_t* seqs, int32_t n_seqs, const int32_t* ids, float* logits_out, int32_t* argmax_out) {
  if (!e || !seqs || !ids) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.decode_step_batch(seqs, n_seqs, ids, logits_out, argmax_out);)
}
int cl_seq_fake_fill(cl_engine* e, cl_seq_t s, int32_t n_tokens) {
  if (!e) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.seq_fake_fill(s, n_tokens);)
}
int cl_debug_kv(cl_engine* e, cl_seq_t s, int32_t layer, int32_t which, int32_t t0, int32_t n, float* out) {
  if (!e || !out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.debug_kv(s, layer, which, t0, n, out);)
}
int cl_time_dominant_kernel(cl_engine* e, cl_seq_t s, int32_t first_id, int32_t n_steps, float* kernel_ms, float* step_ms) {
  if (!e) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  CL_GUARD(return e->impl.time_dominant_kernel(s, first_id, n_steps, kernel_ms, step_ms);)
}
int cl_debug_timeline(cl_engine* e, int64_t* out, int32_t n) {
  if (!e || !out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  return e->impl.debug_timeline(reinterpret_cast<long long*>(out), n);
}
int cl_debug_hidden(cl_engine* e, float* out, int32_t n) {
  if (!e || !out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(e->impl.mu_);
  return e->impl.debug_hidden(out, n);
}

// ---- paged-KV allocator (host logic) ---------------------------------------------------------------
int cl_kvpool_create(int32_t n_pages, int32_t page_size, cl_kvpool** out) {
  if (!out || n_pages <= 0 || page_size <= 0) return CL_ERR_INVALID_ARG;
  *out = new (std::nothrow) cl_kvpool(n_pages, page_size);
  return *out ? CL_OK : CL_ERR_OOM;
}
void cl_kvpool_destroy(cl_kvpool* p) { delete p; }
int cl_kvpool_reserve(cl_kvpool* p, int32_t owner, int32_t n_tokens) {
  if (!p || n_tokens < 0) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(p->mu);
  return p->pool.reserve(owner, n_tokens);
}
int cl_kvpool_release(cl_kvpool* p, int32_t owner) {
  if (!p) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(p->mu);
  return p->pool.release(owner);
}
int cl_kvpool_pages_of(cl_kvpool* p, int32_t owner, int32_t* pages, int32_t cap, int32_t* n_out) {
  if (!p || !n_out) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(p->mu);
  const auto& v = p->pool.pages_of(owner);
  *n_out = (int32_t)v.size();
  if (pages) {
    if (cap < (int32_t)v.size()) return CL_ERR_INVALID_ARG;
    memcpy(pages, v.data(), v.size() * 4);
  }
  return CL_OK;
}
int cl_kvpool_free_pages(cl_kvpool* p) {
  if (!p) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(p->mu);
  return p->pool.free_pages();
}
int cl_kvpool_used_pages(cl_kvpool* p) {
  if (!p) return CL_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lk(p->mu);
  return p->pool.used_pages();
}

}  // extern "C"
