// host_util.cpp — host-side pieces of libclengine.so that need no GPU: paged-KV allocator,
// byte-level tokenizer, sampler, and the minimal protobuf codec for llama.v1.BaseMessage.
#include <algorithm>
#include <cmath>
#include <cstring>

#include "engine.h"

namespace cl {

static thread_local std::string g_last_error;
void set_last_error(const std::string& s) { g_last_error = s; }
const char* get_last_error() { return g_last_error.c_str(); }

// ================================================================================================
// KvPool
// ================================================================================================
KvPool::KvPool(int n_pages, int page_size) : n_pages_(n_pages), page_size_(page_size) {
  free_.reserve(n_pages);
  for (int i = n_pages - 1; i >= 0; --i) free_.push_back(i);
}
int KvPool::reserve(int owner, int n_tokens) {
  auto& v = owned_[owner];
  const int need = (n_tokens + page_size_ - 1) / page_size_;
  const int extra = need - (int)v.size();
  if (extra <= 0) return CL_OK;
  if (extra > (int)free_.size()) return CL_ERR_OOM;
  for (int i = 0; i < extra; ++i) {
    v.push_back(free_.back());
    free_.pop_back();
  }
  return CL_OK;
}
int KvPool::release(int owner) {
  auto it = owned_.find(owner);
  if (it == owned_.end()) return CL_OK;
  for (auto rit = it->second.rbegin(); rit != it->second.rend(); ++rit) free_.push_back(*rit);
  owned_.erase(it);
  return CL_OK;
}
const std::vector<int>& KvPool::pages_of(int owner) {
  auto it = owned_.find(owner);
  return it == owned_.end() ? empty_ : it->second;
}

// ================================================================================================
// Tokenizer (byte-level fallback)
// ================================================================================================
std::vector<int32_t> ByteTokenizer::encode(const std::string& text, bool add_bos) const {
  std::vector<int32_t> ids;
  ids.reserve(text.size() + 1);
  if (add_bos) ids.push_back(bos());
  for (unsigned char c : text) {
    int id = 3 + (int)c;
    if (id >= vocab_) id = 3 + ((int)c % std::max(1, vocab_ - 3));
    ids.push_back(id);
  }
  return ids;
}
std::string ByteTokenizer::decode_bytes(const std::vector<int32_t>& ids) const {
  std::string out;
  for (int32_t id : ids) {
    if (id >= 3 && id < 259) out.push_back((char)(id - 3));
    else if (id < 3) continue;  // specials render as nothing
    else {
      // ids beyond the byte range have no surface form without a vocab file: keep them visible
      // and 7-bit clean so the JSON the gateway emits stays valid UTF-8.
      char buf[24];
      snprintf(buf, sizeof buf, "<%d>", id);
      out += buf;
    }
  }
  return out;
}
// bytes produced by a random-weight model are not valid UTF-8 in general: sanitise
std::string Tokenizer::sanitize(const std::string& out) {
  std::string clean;
  clean.reserve(out.size());
  for (size_t i = 0; i < out.size();) {
    unsigned char c = (unsigned char)out[i];
    int n = c < 0x80 ? 1 : (c >> 5) == 6 ? 2 : (c >> 4) == 14 ? 3 : (c >> 3) == 30 ? 4 : 0;
    bool ok = n > 0 && i + n <= out.size();
    for (int k = 1; ok && k < n; ++k) ok = (((unsigned char)out[i + k]) >> 6) == 2;
    if (ok && n == 1 && c < 0x20 && c != '\n' && c != '\t' && c != '\r') ok = false;
    if (ok) { clean.append(out, i, n); i += n; }
    else { clean += "\xEF\xBF\xBD"; i += 1; }
  }
  return clean;
}
std::string ByteTokenizer::apply_chat_template(const std::string& user_prompt) const {
  return "<|user|>\n" + user_prompt + "\n<|assistant|>\n";
}

// ================================================================================================
// Sampler (same chain and RNG as oracle oc_sample, so identical logits give identical tokens)
// ================================================================================================
static inline uint64_t mix64h(uint64_t x) {
  x ^= x >> 30; x *= 0xBF58476D1CE4E5B9ull;
  x ^= x >> 27; x *= 0x94D049BB133111EBull;
  x ^= x >> 31;
  return x;
}
static double uniform01(uint64_t seed, uint64_t step) {
  uint64_t x = mix64h(seed * 0x9E3779B97F4A7C15ull + step + 0x632BE59BD9B4E019ull);
  return (double)(x >> 11) * (1.0 / 9007199254740992.0);
}
// HF transformers modeling_rope_utils.py, _compute_llama3_parameters (Llama-3.1 / 3.2): wavelengths beyond
// original_max_pos / low_freq_factor are stretched by `factor`, those below original_max_pos / high_freq_factor are kept,
// the band in between is blended linearly.
double rope_inv_freq(const cl_model_config& c, int i) {
  const double pi = 3.14159265358979323846;
  const double inv = std::pow((double)c.rope_theta, -2.0 * (double)i / (double)c.head_dim);
  if (!(c.rope_factor > 1.0f) || c.rope_original_max_pos <= 0) return inv;
  const double factor = c.rope_factor, lo = c.rope_low_freq_factor, hi = c.rope_high_freq_factor, old = c.rope_original_max_pos;
  const double wavelen = 2.0 * pi / inv;
  if (wavelen > old / lo) return inv / factor;
  if (wavelen < old / hi) return inv;
  const double smooth = (old / wavelen - lo) / (hi - lo);
  return (1.0 - smooth) * inv / factor + smooth * inv;
}

int32_t sample_token(const float* logits, int32_t vocab, const cl_sampling& sp, const int32_t* history, int32_t n_history,
                     uint64_t step) {
  if (sp.temperature <= 0.f) {
    int best = 0;
    for (int i = 1; i < vocab; ++i) if (logits[i] > logits[best]) best = i;
    return best;
  }
  struct Cand { float v; int32_t id; };
  std::vector<Cand> c(vocab);
  for (int i = 0; i < vocab; ++i) c[i] = {logits[i], i};
  if (sp.repeat_penalty != 1.0f && sp.repeat_last_n != 0 && history) {
    int start = sp.repeat_last_n > 0 && n_history > sp.repeat_last_n ? n_history - sp.repeat_last_n : 0;
    std::vector<char> seen(vocab, 0);
    for (int i = start; i < n_history; ++i) {
      int id = history[i];
      if (id < 0 || id >= vocab || seen[id]) continue;
      seen[id] = 1;
      c[id].v = c[id].v > 0.f ? c[id].v / sp.repeat_penalty : c[id].v * sp.repeat_penalty;
    }
  }
  auto cmp = [](const Cand& a, const Cand& b) { return a.v > b.v || (a.v == b.v && a.id < b.id); };
  int n = vocab;
  if (sp.top_k > 0 && sp.top_k < n) n = sp.top_k;
  if (n < vocab) std::partial_sort(c.begin(), c.begin() + n, c.end(), cmp);
  else std::sort(c.begin(), c.end(), cmp);
  const float mx = c[0].v;
  std::vector<double> p(n);
  double den = 0.0;
  for (int i = 0; i < n; ++i) { p[i] = std::exp((double)(c[i].v - mx) / (double)sp.temperature); den += p[i]; }
  int keep = n;
  if (sp.top_p > 0.f && sp.top_p < 1.f) {
    double cum = 0.0;
    for (int i = 0; i < n; ++i) { cum += p[i] / den; if (cum >= (double)sp.top_p) { keep = i + 1; break; } }
  }
  double tot = 0.0;
  for (int i = 0; i < keep; ++i) tot += p[i];
  const double u = uniform01(sp.seed, step) * tot;
  double cum = 0.0;
  int32_t pick = c[keep - 1].id;
  for (int i = 0; i < keep; ++i) { cum += p[i]; if (u < cum) { pick = c[i].id; break; } }
  return pick;
}

// ================================================================================================
// protobuf codec.  crowdllama-pb (go.mod:6) is not vendored, so field NUMBERS are an assumption
// kept in this one table (declaration order of the Go struct literals at api.go:77-85,193-197):
//   BaseMessage      { oneof message { GenerateRequest generate_request = 1;
//                                       GenerateResponse generate_response = 2; } }
//   GenerateRequest  { string model = 1; string prompt = 2; bool stream = 3;
//                      GenerateOptions options = 4; }                       <- EXTENSION (SURVEY.md §8f row 3)
//   GenerateOptions  { optional uint64 seed = 1; optional float temperature = 2; optional int32 top_k = 3;
//                      optional float top_p = 4; optional float repeat_penalty = 5;
//                      optional int32 repeat_last_n = 6; optional int32 num_predict = 7; optional bool raw = 8;
//                      optional bool logprobs = 9; optional int32 top_logprobs = 10; }        <- EXTENSION
//   GenerateResponse { string model = 1; google.protobuf.Timestamp created_at = 2;
//                      string response = 3; bool done = 4; string done_reason = 5;
//                      string worker_id = 6; int64 total_duration = 7;
//                      repeated TokenLogprob logprobs = 8; }                                 <- EXTENSION
//   TokenLogprob     { bytes token = 1; float logprob = 2; repeated TopLogprob top_logprobs = 3; }
//   TopLogprob       { bytes token = 1; float logprob = 2; }
// ================================================================================================
enum { kReqOptions = 4, kOptSeed = 1, kOptTemperature = 2, kOptTopK = 3, kOptTopP = 4, kOptRepeatPenalty = 5, kOptRepeatLastN = 6,
       kOptNumPredict = 7, kOptRaw = 8, kOptLogprobs = 9, kOptTopLogprobs = 10 };
enum { kBaseReq = 1, kBaseResp = 2, kReqModel = 1, kReqPrompt = 2, kReqStream = 3, kRespModel = 1, kRespCreated = 2,
       kRespResponse = 3, kRespDone = 4, kRespDoneReason = 5, kRespWorkerId = 6, kRespTotalDuration = 7, kRespLogprobs = 8,
       kLpToken = 1, kLpLogprob = 2, kLpTop = 3 };

static bool rd_varint(const uint8_t*& p, const uint8_t* end, uint64_t* v) {
  uint64_t r = 0;
  for (int shift = 0; shift < 64 && p < end; shift += 7) {
    uint8_t b = *p++;
    r |= (uint64_t)(b & 0x7f) << shift;
    if (!(b & 0x80)) { *v = r; return true; }
  }
  return false;
}
static bool skip_field(const uint8_t*& p, const uint8_t* end, int wt) {
  uint64_t v;
  switch (wt) {
    case 0: return rd_varint(p, end, &v);
    case 1: if (end - p < 8) return false; p += 8; return true;
    case 2: if (!rd_varint(p, end, &v) || (uint64_t)(end - p) < v) return false; p += v; return true;
    case 5: if (end - p < 4) return false; p += 4; return true;
    default: return false;
  }
}
static bool decode_options(const uint8_t* q, const uint8_t* qe, PbGenerateOptions* o) {
  while (q < qe) {
    uint64_t k;
    if (!rd_varint(q, qe, &k)) return false;
    const int f = (int)(k >> 3), wt = (int)(k & 7);
    if (wt == 0 && (f == kOptSeed || f == kOptTopK || f == kOptRepeatLastN || f == kOptNumPredict || f == kOptRaw || f == kOptLogprobs ||
                    f == kOptTopLogprobs)) {
      uint64_t v;
      if (!rd_varint(q, qe, &v)) return false;
      if (f == kOptSeed) o->seed = v;
      else if (f == kOptTopK) o->top_k = (int32_t)(int64_t)v;
      else if (f == kOptRepeatLastN) o->repeat_last_n = (int32_t)(int64_t)v;
      else if (f == kOptNumPredict) o->num_predict = (int32_t)(int64_t)v;
      else if (f == kOptLogprobs) o->logprobs = v != 0;
      else if (f == kOptTopLogprobs) o->top_logprobs = (int32_t)(int64_t)v;
      else o->raw = v != 0;
      o->has |= 1u << f;
    } else if (wt == 5 && (f == kOptTemperature || f == kOptTopP || f == kOptRepeatPenalty)) {
      if (qe - q < 4) return false;
      float v;
      memcpy(&v, q, 4);
      q += 4;
      if (f == kOptTemperature) o->temperature = v; else if (f == kOptTopP) o->top_p = v; else o->repeat_penalty = v;
      o->has |= 1u << f;
    } else if (!skip_field(q, qe, wt)) return false;
  }
  return true;
}
void apply_options(const PbGenerateOptions& o, cl_sampling* sp) {
  if (o.has & (1u << kOptSeed)) sp->seed = o.seed;
  if (o.has & (1u << kOptTemperature)) sp->temperature = o.temperature;
  if (o.has & (1u << kOptTopK)) sp->top_k = o.top_k;
  if (o.has & (1u << kOptTopP)) sp->top_p = o.top_p;
  if (o.has & (1u << kOptRepeatPenalty)) sp->repeat_penalty = o.repeat_penalty;
  if (o.has & (1u << kOptRepeatLastN)) sp->repeat_last_n = o.repeat_last_n;
  if (o.has & (1u << kOptNumPredict)) sp->max_new_tokens = o.num_predict;
}
bool pb_decode_request(const uint8_t* data, size_t len, PbGenerateRequest* out) {
  const uint8_t* p = data; const uint8_t* end = data + len;
  bool found = false;
  while (p < end) {
    uint64_t key;
    if (!rd_varint(p, end, &key)) return false;
    int field = (int)(key >> 3), wt = (int)(key & 7);
    if (field == kBaseReq && wt == 2) {
      uint64_t n;
      if (!rd_varint(p, end, &n) || (uint64_t)(end - p) < n) return false;
      const uint8_t* q = p; const uint8_t* qe = p + n;
      p += n;
      *out = PbGenerateRequest();
      found = true;
      while (q < qe) {
        uint64_t k2;
        if (!rd_varint(q, qe, &k2)) return false;
        int f2 = (int)(k2 >> 3), w2 = (int)(k2 & 7);
        if ((f2 == kReqModel || f2 == kReqPrompt) && w2 == 2) {
          uint64_t m;
          if (!rd_varint(q, qe, &m) || (uint64_t)(qe - q) < m) return false;
          (f2 == kReqModel ? out->model : out->prompt).assign((const char*)q, m);
          q += m;
        } else if (f2 == kReqStream && w2 == 0) {
          uint64_t v;
          if (!rd_varint(q, qe, &v)) return false;
          out->stream = v != 0;
        } else if (f2 == kReqOptions && w2 == 2) {
          uint64_t m;
          if (!rd_varint(q, qe, &m) || (uint64_t)(qe - q) < m) return false;
          if (!decode_options(q, q + m, &out->opt)) return false;
          q += m;
        } else if (!skip_field(q, qe, w2)) return false;
      }
    } else if (!skip_field(p, end, wt)) return false;
  }
  return found;
}
static void wr_varint(std::vector<uint8_t>& b, uint64_t v) {
  while (v >= 0x80) { b.push_back((uint8_t)(v | 0x80)); v >>= 7; }
  b.push_back((uint8_t)v);
}
static void wr_str(std::vector<uint8_t>& b, int field, const std::string& s) {
  if (s.empty()) return;  // proto3: default values are not serialised
  wr_varint(b, (uint64_t)field << 3 | 2);
  wr_varint(b, s.size());
  b.insert(b.end(), s.begin(), s.end());
}
static void wr_i64(std::vector<uint8_t>& b, int field, int64_t v) {
  if (!v) return;
  wr_varint(b, (uint64_t)field << 3 | 0);
  wr_varint(b, (uint64_t)v);
}
static void wr_f32(std::vector<uint8_t>& b, int field, float v) {
  if (v == 0.f) return;
  wr_varint(b, (uint64_t)field << 3 | 5);
  uint8_t x[4];
  memcpy(x, &v, 4);
  b.insert(b.end(), x, x + 4);
}
static void wr_msg(std::vector<uint8_t>& b, int field, const std::vector<uint8_t>& m) {   // present even when empty
  wr_varint(b, (uint64_t)field << 3 | 2);
  wr_varint(b, m.size());
  b.insert(b.end(), m.begin(), m.end());
}
std::vector<uint8_t> pb_encode_response(const PbGenerateResponse& r) {
  std::vector<uint8_t> ts;
  wr_i64(ts, 1, r.created_at_sec);
  wr_i64(ts, 2, r.created_at_nanos);
  std::vector<uint8_t> in;
  wr_str(in, kRespModel, r.model);
  if (!ts.empty()) {
    wr_varint(in, (uint64_t)kRespCreated << 3 | 2);
    wr_varint(in, ts.size());
    in.insert(in.end(), ts.begin(), ts.end());
  }
  wr_str(in, kRespResponse, r.response);
  wr_i64(in, kRespDone, r.done ? 1 : 0);
  wr_str(in, kRespDoneReason, r.done_reason);
  wr_str(in, kRespWorkerId, r.worker_id);
  wr_i64(in, kRespTotalDuration, r.total_duration);
  for (const auto& t : r.logprobs) {
    std::vector<uint8_t> m;
    wr_str(m, kLpToken, t.token);
    wr_f32(m, kLpLogprob, t.logprob);
    for (const auto& a : t.top_logprobs) {
      std::vector<uint8_t> n;
      wr_str(n, kLpToken, a.token);
      wr_f32(n, kLpLogprob, a.logprob);
      wr_msg(m, kLpTop, n);
    }
    wr_msg(in, kRespLogprobs, m);
  }
  std::vector<uint8_t> out;
  wr_varint(out, (uint64_t)kBaseResp << 3 | 2);
  wr_varint(out, in.size());
  out.insert(out.end(), in.begin(), in.end());
  return out;
}

}  // namespace cl
