// tokenizer.cpp — native tokenizer for HF `tokenizer.json` files (SURVEY.md §8f row 2).
//
// Upstream of the reference's handler the Ollama server tokenises with the model's own vocabulary (llama.cpp
// llama-vocab: SentencePiece-BPE for Llama-2 / Mistral / TinyLlama, tiktoken-style byte-level BPE for Llama-3;
// call site /root/reference/pkg/crowdllama/api.go:108-160).  No vocabulary file exists offline, so this loader is
// pinned against the HF `tokenizers` library instead: tests/golden/make_tokenizer_golden.py trains three small
// tokenizers with exactly the pipeline components those families ship and records ids + decoded text for 31 strings
// each; tests/test_tokenizer.py requires identical output.  Supported pipeline:
//   added tokens       leftmost-longest match on the raw text (chat markers, <s>, </s>, ...)
//   normalizer         null | Prepend | Replace(String) | Sequence of those
//   pre_tokenizer      null | Metaspace | ByteLevel | Split(regex) + ByteLevel   (GPT-2 and Llama-3 regex flavours,
//                      implemented as hand-written scanners; Unicode classes \p{L} \p{N} from generated range tables
//                      (unicode_tables.inc), \s = the White_Space property)
//   model              BPE: vocab, merges ("a b" or [a, b]), byte_fallback, ignore_merges, unk_token
//   decoder            ByteLevel | SentencePiece chain (Replace ▁, ByteFallback, Fuse, Strip)
#include <algorithm>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <queue>
#include <sstream>
#include <unordered_map>

#include "engine.h"
#include "json_min.h"

namespace cl {

namespace {
using jsonmin::JVal;
using jsonmin::JParser;
using jsonmin::append_utf8;


// ================================================================================================
// UTF-8 and Unicode classes
// ================================================================================================
// decodes one code point; invalid bytes come back as themselves (length 1)
uint32_t next_cp(const std::string& s, size_t i, int* len) {
  const unsigned char c = (unsigned char)s[i];
  int n = c < 0x80 ? 1 : (c >> 5) == 6 ? 2 : (c >> 4) == 14 ? 3 : (c >> 3) == 30 ? 4 : 1;
  if (i + n > s.size()) n = 1;
  for (int k = 1; k < n; ++k) if ((((unsigned char)s[i + k]) >> 6) != 2) { n = 1; break; }
  *len = n;
  if (n == 1) return c;
  uint32_t cp = n == 2 ? (c & 0x1F) : n == 3 ? (c & 0x0F) : (c & 0x07);
  for (int k = 1; k < n; ++k) cp = (cp << 6) | (((unsigned char)s[i + k]) & 0x3F);
  return cp;
}

struct Range { uint32_t lo, hi; };
bool in_ranges(uint32_t cp, const Range* r, size_t n) {
  size_t lo = 0, hi = n;
  while (lo < hi) {
    const size_t mid = (lo + hi) / 2;
    if (cp < r[mid].lo) hi = mid; else if (cp > r[mid].hi) lo = mid + 1; else return true;
  }
  return false;
}
#include "unicode_tables.inc"   // kLetters / kNumbers: exact \\p{L} and \\p{N} ranges (tools/gen_unicode_tables.py)
bool is_letter(uint32_t cp) { return in_ranges(cp, kLetters, sizeof kLetters / sizeof *kLetters); }
bool is_number(uint32_t cp) { return in_ranges(cp, kNumbers, sizeof kNumbers / sizeof *kNumbers); }
bool is_space(uint32_t cp) {
  return (cp >= 0x09 && cp <= 0x0D) || cp == 0x20 || cp == 0x85 || cp == 0xA0 || cp == 0x1680 || (cp >= 0x2000 && cp <= 0x200A) ||
         cp == 0x2028 || cp == 0x2029 || cp == 0x202F || cp == 0x205F || cp == 0x3000;
}
bool is_newline(uint32_t cp) { return cp == '\n' || cp == '\r'; }

struct Cp { uint32_t cp; uint32_t off; };   // code point + byte offset
std::vector<Cp> code_points(const std::string& s) {
  std::vector<Cp> v;
  v.reserve(s.size() + 1);
  for (size_t i = 0; i < s.size();) {
    int n;
    const uint32_t cp = next_cp(s, i, &n);
    v.push_back({cp, (uint32_t)i});
    i += n;
  }
  v.push_back({0, (uint32_t)s.size()});   // sentinel
  return v;
}

// ---- regex flavours as scanners: return the end (index into cps) of the piece starting at i ----------------------
// Llama-3: (?i:'s|'t|'re|'ve|'m|'ll|'d)|[^\r\n\p{L}\p{N}]?\p{L}+|\p{N}{1,3}| ?[^\s\p{L}\p{N}]+[\r\n]*|\s*[\r\n]+|\s+(?!\S)|\s+
// GPT-2:   's|'t|'re|'ve|'m|'ll|'d| ?\p{L}+| ?\p{N}+| ?[^\s\p{L}\p{N}]+|\s+(?!\S)|\s+
size_t scan_piece(const std::vector<Cp>& c, size_t i, bool llama3) {
  const size_t n = c.size() - 1;
  auto lower = [](uint32_t x) { return x >= 'A' && x <= 'Z' ? x + 32 : x; };
  auto other = [](uint32_t x) { return !is_space(x) && !is_letter(x) && !is_number(x); };
  const uint32_t a = c[i].cp;
  if (a == '\'' && i + 1 < n) {   // contractions
    const uint32_t b1 = llama3 ? lower(c[i + 1].cp) : c[i + 1].cp, b2 = i + 2 < n ? (llama3 ? lower(c[i + 2].cp) : c[i + 2].cp) : 0;
    if (b1 == 's' || b1 == 't' || b1 == 'm' || b1 == 'd') return i + 2;
    if ((b1 == 'r' && b2 == 'e') || (b1 == 'v' && b2 == 'e') || (b1 == 'l' && b2 == 'l')) return i + 3;
  }
  if (llama3) {
    // [^\r\n\p{L}\p{N}]?\p{L}+
    {
      size_t j = i;
      if (!is_newline(a) && !is_letter(a) && !is_number(a) && i + 1 < n && is_letter(c[i + 1].cp)) j = i + 1;
      if (is_letter(c[j].cp) && j < n) {
        while (j < n && is_letter(c[j].cp)) ++j;
        return j;
      }
    }
    // \p{N}{1,3}
    if (is_number(a)) {
      size_t j = i;
      while (j < n && j < i + 3 && is_number(c[j].cp)) ++j;
      return j;
    }
    //  ?[^\s\p{L}\p{N}]+[\r\n]*
    {
      size_t j = i;
      if (a == ' ' && i + 1 < n && other(c[i + 1].cp)) j = i + 1;
      if (j < n && other(c[j].cp)) {
        while (j < n && other(c[j].cp)) ++j;
        while (j < n && is_newline(c[j].cp)) ++j;
        return j;
      }
    }
  } else {
    size_t j = i;
    if (a == ' ' && i + 1 < n) j = i + 1;
    if (j < n && is_letter(c[j].cp)) { while (j < n && is_letter(c[j].cp)) ++j; return j; }
    if (j < n && is_number(c[j].cp)) { while (j < n && is_number(c[j].cp)) ++j; return j; }
    if (j < n && other(c[j].cp)) { while (j < n && other(c[j].cp)) ++j; return j; }
  }
  // whitespace alternatives
  size_t run = i;
  while (run < n && is_space(c[run].cp)) ++run;
  if (run == i) return i + 1;   // defensive: a character no alternative claims
  if (llama3) {                  // \s*[\r\n]+ : up to and including the last newline of the run
    size_t last_nl = 0; bool has = false;
    for (size_t j = i; j < run; ++j) if (is_newline(c[j].cp)) { last_nl = j; has = true; }
    if (has) return last_nl + 1;
  }
  if (run == n) return run;            // \s+(?!\S) at the end of the text
  if (run - i >= 2) return run - 1;    // \s+(?!\S): leave the last space to the next piece
  return run;                          // \s+
}

// GPT-2 byte <-> unicode table
struct ByteMap {
  uint32_t to_cp[256];
  std::unordered_map<uint32_t, uint8_t> to_byte;
  ByteMap() {
    int extra = 0;
    for (int b = 0; b < 256; ++b) {
      const bool keep = (b >= 33 && b <= 126) || (b >= 161 && b <= 172) || (b >= 174 && b <= 255);
      to_cp[b] = keep ? (uint32_t)b : 256u + (uint32_t)extra++;
      to_byte[to_cp[b]] = (uint8_t)b;
    }
  }
};
const ByteMap& byte_map() { static const ByteMap m; return m; }

const char kMeta[] = "\xE2\x96\x81";   // U+2581 "▁"

void replace_all(std::string& s, const std::string& from, const std::string& to) {
  if (from.empty()) return;
  size_t pos = 0;
  while ((pos = s.find(from, pos)) != std::string::npos) { s.replace(pos, from.size(), to); pos += to.size(); }
}

}  // namespace

// ================================================================================================
// HfBpeTokenizer
// ================================================================================================
class HfBpeTokenizer : public Tokenizer {
 public:
  bool load(const std::string& path, const std::string& chat_family, std::string* err);
  std::vector<int32_t> encode(const std::string& text, bool add_bos) const override;
  std::string decode_bytes(const std::vector<int32_t>& ids) const override;
  std::string token_bytes(int id) const override {
    if (id >= 0 && id < (int)id_to_tok_.size() && special_[id]) return id_to_tok_[id];   // added-token content
    return decode_bytes({id});
  }
  int bos() const override { return bos_; }
  int eos() const override { return eos_; }
  bool is_stop(int id) const override { return id == eos_ || id == eot_; }
  std::string apply_chat_template(const std::string& user_prompt) const override;
  int vocab_size() const override { return (int)id_to_tok_.size(); }

 private:
  struct NormStep { int kind; std::string a, b; };   // 0 = Prepend(a), 1 = Replace(a -> b)
  std::vector<NormStep> norm_;
  bool byte_level_ = false, llama3_regex_ = false, use_regex_ = false, metaspace_ = false, meta_split_ = false, bl_prefix_space_ = false;
  int meta_prepend_ = 0;                              // 0 never, 1 first, 2 always
  bool byte_fallback_ = false, ignore_merges_ = false, spm_decoder_ = false, strip_leading_space_ = false;
  std::unordered_map<std::string, int> vocab_;
  std::vector<std::string> id_to_tok_;
  std::vector<char> special_;                         // id -> skipped on decode
  std::vector<char> is_added_;                        // id -> added token (surface form = content, not byte-level mapped)
  bool added_first_[256] = {};                        // bytes that can start an added token
  std::unordered_map<uint64_t, std::pair<int, int>> merges_;   // (a << 32 | b) -> (rank, merged id)
  std::vector<std::pair<std::string, int>> added_;    // content, id (sorted by length desc)
  int unk_ = -1, bos_ = -1, eos_ = -1, eot_ = -1, byte_tok_[256];
  std::string family_;

  void bpe_word(const std::string& w, std::vector<int32_t>* out) const;
  void encode_segment(const std::string& seg, bool first, std::vector<int32_t>* out) const;
  int find(const char* t) const { auto it = vocab_.find(t); return it == vocab_.end() ? -1 : it->second; }
};

bool HfBpeTokenizer::load(const std::string& path, const std::string& chat_family, std::string* err) {
  std::ifstream f(path, std::ios::binary);
  if (!f) { *err = "cannot open " + path; return false; }
  std::stringstream ss;
  ss << f.rdbuf();
  const std::string text = ss.str();
  JVal root;
  JParser jp{text.data(), text.data() + text.size(), {}};
  if (!jp.value(&root) || root.type != JVal::Obj) { *err = "tokenizer.json: " + (jp.err.empty() ? std::string("not an object") : jp.err); return false; }
  const JVal* model = root.get("model");
  if (!model || model->str("type", "BPE") != "BPE" || !model->get("vocab")) { *err = "tokenizer.json: only BPE models are supported"; return false; }
  for (auto& kv : model->get("vocab")->o) {
    const int id = (int)kv.second.n;
    vocab_[kv.first] = id;
    if ((int)id_to_tok_.size() <= id) id_to_tok_.resize(id + 1);
    id_to_tok_[id] = kv.first;
  }
  byte_fallback_ = model->boolean("byte_fallback", false);
  ignore_merges_ = model->boolean("ignore_merges", false);
  unk_ = find(model->str("unk_token", "").c_str());
  // added tokens
  if (const JVal* at = root.get("added_tokens")) {
    for (auto& t : at->a) {
      const JVal* idv = t.get("id");
      const std::string& content = t.str("content", "");
      if (!idv || content.empty()) continue;
      const int id = (int)idv->n;
      vocab_[content] = id;
      if ((int)id_to_tok_.size() <= id) id_to_tok_.resize(id + 1);
      id_to_tok_[id] = content;
      added_.emplace_back(content, id);
      if (t.boolean("special", false)) { special_.resize(std::max(special_.size(), (size_t)id + 1), 0); special_[id] = 1; }
    }
    std::sort(added_.begin(), added_.end(), [](auto& x, auto& y) { return x.first.size() > y.first.size(); });
  }
  special_.resize(id_to_tok_.size(), 0);
  is_added_.assign(id_to_tok_.size(), 0);
  for (auto& at : added_) { is_added_[at.second] = 1; added_first_[(unsigned char)at.first[0]] = true; }
  // merges
  if (const JVal* mg = model->get("merges")) {
    int rank = 0;
    for (auto& m : mg->a) {
      std::string a, b;
      if (m.type == JVal::Arr && m.a.size() == 2) { a = m.a[0].s; b = m.a[1].s; }
      else if (m.type == JVal::Str) { const size_t sp = m.s.find(' '); if (sp == std::string::npos) continue; a = m.s.substr(0, sp); b = m.s.substr(sp + 1); }
      const int ia = find(a.c_str()), ib = find(b.c_str()), ic = find((a + b).c_str());
      if (ia >= 0 && ib >= 0 && ic >= 0) merges_.emplace(((uint64_t)(uint32_t)ia << 32) | (uint32_t)ib, std::make_pair(rank, ic));
      ++rank;
    }
  }
  for (int b = 0; b < 256; ++b) {
    char name[8];
    snprintf(name, sizeof name, "<0x%02X>", b);
    byte_tok_[b] = find(name);
    if (byte_tok_[b] < 0) byte_fallback_ = false;   // byte fallback needs all 256 <0xXX> tokens
  }
  // normalizer
  std::vector<const JVal*> steps;
  if (const JVal* nz = root.get("normalizer")) {
    if (nz->type == JVal::Obj) {
      if (nz->str("type", "") == "Sequence" && nz->get("normalizers")) for (auto& x : nz->get("normalizers")->a) steps.push_back(&x);
      else steps.push_back(nz);
    }
  }
  for (const JVal* st : steps) {
    const std::string& ty = st->str("type", "");
    if (ty == "Prepend") norm_.push_back({0, st->str("prepend", ""), ""});
    else if (ty == "Replace" && st->get("pattern") && st->get("pattern")->get("String"))
      norm_.push_back({1, st->get("pattern")->get("String")->s, st->str("content", "")});
    // NFC / NFKC / Lowercase ...: not applied (none of the target families uses them)
  }
  // pre-tokenizer
  std::vector<const JVal*> pts;
  if (const JVal* pt = root.get("pre_tokenizer")) {
    if (pt->type == JVal::Obj) {
      if (pt->str("type", "") == "Sequence" && pt->get("pretokenizers")) for (auto& x : pt->get("pretokenizers")->a) pts.push_back(&x);
      else pts.push_back(pt);
    }
  }
  for (const JVal* pt : pts) {
    const std::string& ty = pt->str("type", "");
    if (ty == "ByteLevel") {
      byte_level_ = true;
      bl_prefix_space_ = pt->boolean("add_prefix_space", false);
      if (pt->boolean("use_regex", true)) use_regex_ = true;            // GPT-2 regex inside ByteLevel
    } else if (ty == "Split") {
      use_regex_ = true;
      const JVal* pat = pt->get("pattern");
      const std::string rx = pat && pat->get("Regex") ? pat->get("Regex")->s : "";
      llama3_regex_ = rx.find("\\p{N}{1,3}") != std::string::npos;
    } else if (ty == "Metaspace") {
      metaspace_ = true;
      meta_split_ = pt->boolean("split", true);
      const std::string& sch = pt->str("prepend_scheme", "always");
      meta_prepend_ = sch == "never" ? 0 : sch == "first" ? 1 : 2;
      if (const JVal* aps = pt->get("add_prefix_space")) if (aps->type == JVal::Bool && !aps->b) meta_prepend_ = 0;
    }
  }
  // decoder
  if (const JVal* dc = root.get("decoder")) {
    if (dc->type == JVal::Obj && dc->str("type", "") != "ByteLevel") {
      spm_decoder_ = true;
      if (dc->get("decoders")) for (auto& d : dc->get("decoders")->a) if (d.str("type", "") == "Strip" && d.get("start") && d.get("start")->n >= 1) strip_leading_space_ = true;
      if (dc->str("type", "") == "Metaspace") strip_leading_space_ = true;
    }
  }
  // special ids and chat family
  bos_ = find("<|begin_of_text|>"); if (bos_ < 0) bos_ = find("<s>"); if (bos_ < 0) bos_ = find("<|startoftext|>");
  eos_ = find("<|end_of_text|>"); if (eos_ < 0) eos_ = find("</s>"); if (eos_ < 0) eos_ = find("<|endoftext|>");
  eot_ = find("<|eot_id|>"); if (eot_ < 0) eot_ = find("<|im_end|>");
  family_ = chat_family;
  if (family_.empty()) {
    if (find("<|start_header_id|>") >= 0) family_ = "llama3";
    else if (find("<|im_start|>") >= 0) family_ = "chatml";
    else if (find("[INST]") >= 0) family_ = "mistral";
    else if (find("<|user|>") >= 0) family_ = "zephyr";
    else family_ = "mistral";
  }
  if (id_to_tok_.empty()) { *err = "tokenizer.json: empty vocabulary"; return false; }
  return true;
}

// BPE over one pre-tokenised word (already normalised / byte-level mapped)
void HfBpeTokenizer::bpe_word(const std::string& w, std::vector<int32_t>* out) const {
  if (w.empty()) return;
  if (ignore_merges_) {
    auto it = vocab_.find(w);
    if (it != vocab_.end()) { out->push_back(it->second); return; }
  }
  // symbols: one per character (known), bytes (fallback) or unk
  struct Sym { int id; int prev, next; };
  std::vector<Sym> sym;
  bool last_unk = false;
  for (size_t i = 0; i < w.size();) {
    int n;
    next_cp(w, i, &n);
    const std::string ch = w.substr(i, n);
    auto it = vocab_.find(ch);
    if (it != vocab_.end()) { sym.push_back({it->second, 0, 0}); last_unk = false; }
    else if (byte_fallback_) { for (int k = 0; k < n; ++k) sym.push_back({byte_tok_[(unsigned char)ch[k]], 0, 0}); last_unk = false; }
    else if (unk_ >= 0) { if (!last_unk) sym.push_back({unk_, 0, 0}); last_unk = true; }   // fuse_unk
    i += n;
  }
  const int n = (int)sym.size();
  for (int i = 0; i < n; ++i) { sym[i].prev = i - 1; sym[i].next = i + 1 < n ? i + 1 : -1; }
  struct Cand { int rank, pos, left_id, right_id, merged; };
  auto cmp = [](const Cand& a, const Cand& b) { return a.rank != b.rank ? a.rank > b.rank : a.pos > b.pos; };
  std::priority_queue<Cand, std::vector<Cand>, decltype(cmp)> pq(cmp);
  auto push = [&](int i) {
    if (i < 0 || sym[i].next < 0) return;
    const int j = sym[i].next;
    auto it = merges_.find(((uint64_t)(uint32_t)sym[i].id << 32) | (uint32_t)sym[j].id);
    if (it != merges_.end()) pq.push({it->second.first, i, sym[i].id, sym[j].id, it->second.second});
  };
  for (int i = 0; i < n; ++i) push(i);
  while (!pq.empty()) {
    const Cand c = pq.top();
    pq.pop();
    const int i = c.pos;
    if (sym[i].id != c.left_id || sym[i].next < 0 || sym[sym[i].next].id != c.right_id) continue;   // stale
    const int j = sym[i].next;
    sym[i].id = c.merged;
    sym[i].next = sym[j].next;
    if (sym[j].next >= 0) sym[sym[j].next].prev = i;
    sym[j].id = -1;
    push(sym[i].prev);
    push(i);
  }
  for (int i = 0; i >= 0 && i < n; i = sym[i].next) out->push_back(sym[i].id);
}

void HfBpeTokenizer::encode_segment(const std::string& seg0, bool first, std::vector<int32_t>* out) const {
  if (seg0.empty()) return;
  std::string seg = seg0;
  for (const NormStep& st : norm_) {
    if (st.kind == 0) { if (!seg.empty()) seg = st.a + seg; }
    else replace_all(seg, st.a, st.b);
  }
  if (metaspace_) {
    replace_all(seg, " ", kMeta);
    const bool starts = seg.compare(0, 3, kMeta) == 0;
    if (!starts && (meta_prepend_ == 2 || (meta_prepend_ == 1 && first))) seg = kMeta + seg;
    if (meta_split_) {   // split before every ▁
      size_t start = 0;
      for (size_t i = 3; i + 3 <= seg.size(); ++i)
        if (seg.compare(i, 3, kMeta) == 0) { bpe_word(seg.substr(start, i - start), out); start = i; i += 2; }
      bpe_word(seg.substr(start), out);
      return;
    }
    bpe_word(seg, out);
    return;
  }
  if (byte_level_) {
    if (bl_prefix_space_ && seg[0] != ' ') seg = " " + seg;
    const ByteMap& bm = byte_map();
    auto emit = [&](size_t b0, size_t b1) {
      std::string w;
      for (size_t i = b0; i < b1; ++i) append_utf8(w, bm.to_cp[(unsigned char)seg[i]]);
      bpe_word(w, out);
    };
    if (!use_regex_) { emit(0, seg.size()); return; }
    const std::vector<Cp> cps = code_points(seg);
    for (size_t i = 0; i + 1 < cps.size();) {
      const size_t j = scan_piece(cps, i, llama3_regex_);
      emit(cps[i].off, cps[j].off);
      i = j;
    }
    return;
  }
  bpe_word(seg, out);
}

std::vector<int32_t> HfBpeTokenizer::encode(const std::string& text, bool add_bos) const {
  std::vector<int32_t> out;
  if (add_bos && bos_ >= 0) out.push_back(bos_);
  size_t seg_start = 0;
  bool first = true;
  for (size_t i = 0; i < text.size();) {
    int hit = -1; size_t hit_len = 0;
    if (!added_first_[(unsigned char)text[i]]) { ++i; continue; }
    for (auto& at : added_)   // sorted by length: the first hit is the longest
      if (at.first.size() <= text.size() - i && text.compare(i, at.first.size(), at.first) == 0) { hit = at.second; hit_len = at.first.size(); break; }
    if (hit < 0) { ++i; continue; }
    encode_segment(text.substr(seg_start, i - seg_start), first && seg_start == 0, &out);
    out.push_back(hit);
    i += hit_len;
    seg_start = i;
    first = false;
  }
  encode_segment(text.substr(seg_start), first && seg_start == 0, &out);
  return out;
}

std::string HfBpeTokenizer::decode_bytes(const std::vector<int32_t>& ids) const {
  std::string out;
  const ByteMap& bm = byte_map();
  for (int32_t id : ids) {
    if (id < 0 || id >= (int)id_to_tok_.size() || special_[id]) continue;
    const std::string& t = id_to_tok_[id];
    if (!spm_decoder_ && byte_level_) {
      if (is_added_[id]) { out += t; continue; }
      for (size_t i = 0; i < t.size();) {
        int n;
        const uint32_t cp = next_cp(t, i, &n);
        auto it = bm.to_byte.find(cp);
        if (it != bm.to_byte.end()) out.push_back((char)it->second); else out.append(t, i, n);
        i += n;
      }
    } else {
      unsigned bv;
      if (t.size() == 6 && t[0] == '<' && t[1] == '0' && t[2] == 'x' && t[5] == '>' && sscanf(t.c_str(), "<0x%02X>", &bv) == 1) out.push_back((char)bv);
      else { std::string piece = t; replace_all(piece, kMeta, " "); out += piece; }
    }
  }
  if (spm_decoder_ && strip_leading_space_ && !out.empty() && out[0] == ' ') out.erase(0, 1);
  return out;
}

std::string HfBpeTokenizer::apply_chat_template(const std::string& p) const {
  // single user turn + generation prompt, as the reference sends it (role forced to "user", api.go:111-116);
  // BOS is added by encode(add_bos = true), not by the template
  if (family_ == "llama3")
    return "<|start_header_id|>user<|end_header_id|>\n\n" + p + "<|eot_id|><|start_header_id|>assistant<|end_header_id|>\n\n";
  if (family_ == "chatml") return "<|im_start|>user\n" + p + "<|im_end|>\n<|im_start|>assistant\n";
  if (family_ == "zephyr") return "<|user|>\n" + p + "</s>\n<|assistant|>\n";
  return "[INST] " + p + " [/INST]";   // mistral-instruct / llama-2-chat without system prompt
}

std::unique_ptr<Tokenizer> load_hf_tokenizer(const std::string& path, const std::string& chat_family, std::string* err) {
  std::unique_ptr<HfBpeTokenizer> t(new HfBpeTokenizer());
  if (!t->load(path, chat_family, err)) return nullptr;
  return t;
}

}  // namespace cl
