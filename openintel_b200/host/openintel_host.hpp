// openintel_host.hpp — C++ host layer above the C ABI (include/openintel_gpu.h), mirroring the
// reference's ports-and-adapters conventions (the reference is Rust; no Rust toolchain exists in the
// build image, so this layer is what a host program links today and what INTEGRATION.md's Rust
// adapter is a transliteration of):
//   DomainError            <- src/domain/error.rs:3-22 (SourceFailure{name, message} for adapter faults)
//   SocialPost, PostSignal <- src/domain/entities/social_post.rs:30-38, src/domain/values/post_signal.rs:3-7
//   PostAnalyzer           <- src/domain/ports/post_analyzer.rs:7-11 (one signal per post, input order)
//   HybridSearch           <- new port in the same shape (the reference has no search port: SURVEY.md §0)
//   tokenize()             <- src/adapters/analyzer/lexicon.rs:54-58
//   IndexBuilder           <- SURVEY.md §8(f) row 1: posts -> vocabulary + CSR postings + doc lengths (host reference)
//   Vocabulary             <- the vocabulary of an index built from text on the device (GpuHybridSearch's text form)
// Header-only; compute happens in libopenintel_gpu.so.  No CPU scoring path exists here either.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <string_view>
#include <unordered_map>
#include <vector>

#include "../../include/openintel_gpu.h"

namespace openintel {

// ---- errors ------------------------------------------------------------------------------------
struct DomainError : std::runtime_error {
  enum Kind { InvalidPostText, AnalyzerMismatch, SourceFailure, NoData };
  Kind kind;
  std::string name;  // SourceFailure: the failing adapter ("gpu-search", "gpu-lexicon")
  DomainError(Kind k, const std::string &n, const std::string &msg) : std::runtime_error(msg), kind(k), name(n) {}
  static DomainError source_failure(const std::string &name, const std::string &message) {
    return DomainError(SourceFailure, name, "data source '" + name + "' failed: " + message);
  }
};

// ---- entities / values ---------------------------------------------------------------------------
struct SocialPost {
  std::string id;
  std::string source;  // "reddit" | "bluesky"
  std::string author;
  std::string text;    // trimmed, non-empty, <= 10 000 chars (PostText)
  int64_t created_at = 0;
  uint32_t engagement = 0;
};
struct PostSignal {
  double polarity = 0.0;  // clamped to [-1, 1]
  bool speculative = false;
};
struct SearchQuery {
  std::vector<float> embedding;  // L2-normalised, index dimension
  std::vector<uint32_t> terms;   // term ids of the index vocabulary
};
struct Hit {
  uint32_t doc_id;
  float rrf;
  uint32_t rank_cosine, rank_bm25;  // 1-based, 0 = absent from that list
};

// ---- ports ---------------------------------------------------------------------------------------
struct PostAnalyzer {
  virtual ~PostAnalyzer() = default;
  // one PostSignal per input post, aligned to input order
  virtual std::vector<PostSignal> analyze(const std::vector<SocialPost> &posts) const = 0;
};
struct HybridSearch {
  virtual ~HybridSearch() = default;
  // one ranked list (RRF desc, doc id asc, <= k hits) per query, aligned to input order
  virtual std::vector<std::vector<Hit>> search(const std::vector<SearchQuery> &queries, size_t k) const = 0;
};

// ---- tokenizer (SPEC §6) -------------------------------------------------------------------------
// Unicode-lowercase, split on every char that is not ASCII alphanumeric, drop empty tokens.  On UTF-8
// bytes: non-ASCII bytes separate, except U+212A KELVIN SIGN -> 'k' and U+0130 -> 'i' + separator.
template <class F>
inline void tokenize(std::string_view text, F &&emit) {
  std::string cur;
  auto flush = [&]() {
    if (!cur.empty()) { emit(std::string_view(cur)); cur.clear(); }
  };
  const size_t n = text.size();
  for (size_t i = 0; i < n;) {
    const unsigned char b = (unsigned char)text[i];
    if (b < 0x80) {
      if (b >= 'A' && b <= 'Z') cur.push_back((char)(b + 32));
      else if ((b >= 'a' && b <= 'z') || (b >= '0' && b <= '9')) cur.push_back((char)b);
      else flush();
      ++i;
    } else if (b == 0xE2 && i + 2 < n && (unsigned char)text[i + 1] == 0x84 && (unsigned char)text[i + 2] == 0xAA) {
      cur.push_back('k');
      i += 3;
    } else if (b == 0xC4 && i + 1 < n && (unsigned char)text[i + 1] == 0xB0) {
      cur.push_back('i');
      flush();
      i += 2;
    } else {
      flush();
      ++i;
    }
  }
  flush();
}
inline std::vector<std::string> tokenize(std::string_view text) {
  std::vector<std::string> out;
  tokenize(text, [&](std::string_view t) { out.emplace_back(t); });
  return out;
}

// query text -> term ids: unknown tokens (term_id gives OI_NO_DOC) dropped, duplicates dropped in first-seen order (SPEC
// §3 counts a term once and scores at most the first 64 DISTINCT known terms; the library de-duplicates too, this keeps
// the arrays small)
template <class TermId>
inline std::vector<uint32_t> query_terms_of(std::string_view text, TermId &&term_id) {
  std::vector<uint32_t> out;
  tokenize(text, [&](std::string_view t) {
    const uint32_t id = term_id(t);
    if (id != OI_NO_DOC && std::find(out.begin(), out.end(), id) == out.end()) out.push_back(id);
  });
  return out;
}

// ---- index builder -------------------------------------------------------------------------------
// Posts in, CSR inverted index out: dense doc ids in input order, exact-token vocabulary (no stemming,
// no stop words: src/domain/dip.rs:261-272 idiom), term ids = lexicographic rank of the token.
class IndexBuilder {
 public:
  void add(std::string_view text) {
    std::vector<uint32_t> toks;
    tokenize(text, [&](std::string_view t) {
      auto it = prov_.find(std::string(t));
      uint32_t id;
      if (it == prov_.end()) {
        id = (uint32_t)terms_.size();
        prov_.emplace(std::string(t), id);
        terms_.emplace_back(t);
      } else {
        id = it->second;
      }
      toks.push_back(id);
    });
    doc_len_.push_back((uint32_t)toks.size());
    std::sort(toks.begin(), toks.end());
    const uint32_t doc = (uint32_t)doc_len_.size() - 1;
    for (size_t i = 0; i < toks.size();) {
      size_t j = i;
      while (j < toks.size() && toks[j] == toks[i]) ++j;
      raw_.push_back({toks[i], doc, (uint32_t)(j - i)});
      i = j;
    }
    finished_ = false;
  }
  void add(const SocialPost &p) {
    ids_.push_back(p.id);
    add(std::string_view(p.text));
  }
  // sorts the vocabulary and lays the postings out as CSR; idempotent
  void finish() {
    if (finished_) return;
    const uint32_t V = (uint32_t)terms_.size();
    std::vector<uint32_t> order(V), rank(V);
    for (uint32_t i = 0; i < V; ++i) order[i] = i;
    std::sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return terms_[a] < terms_[b]; });
    for (uint32_t r = 0; r < V; ++r) rank[order[r]] = r;
    vocab_.resize(V);
    for (uint32_t r = 0; r < V; ++r) vocab_[r] = terms_[order[r]];
    term_off_.assign((size_t)V + 1, 0);
    for (const Raw &p : raw_) ++term_off_[rank[p.term] + 1];
    for (uint32_t t = 0; t < V; ++t) term_off_[t + 1] += term_off_[t];
    doc_ids_.resize(raw_.size());
    tfs_.resize(raw_.size());
    std::vector<uint64_t> cur(term_off_.begin(), term_off_.end() - 1);
    for (const Raw &p : raw_) {  // raw_ is in ascending doc order, so every list comes out ascending
      const uint64_t at = cur[rank[p.term]]++;
      doc_ids_[at] = p.doc;
      tfs_[at] = p.tf;
    }
    finished_ = true;
  }
  uint32_t n_docs() const { return (uint32_t)doc_len_.size(); }
  uint32_t n_terms() const { return (uint32_t)vocab_.size(); }
  const std::vector<uint64_t> &term_offsets() const { return term_off_; }
  const std::vector<uint32_t> &doc_ids() const { return doc_ids_; }
  const std::vector<uint32_t> &tfs() const { return tfs_; }
  const std::vector<uint32_t> &doc_len() const { return doc_len_; }
  const std::vector<std::string> &vocabulary() const { return vocab_; }
  const std::vector<std::string> &post_ids() const { return ids_; }
  // term id of a token, or OI_NO_DOC when the token is not in the vocabulary (contributes 0: SPEC §3)
  uint32_t term_id(std::string_view token) const {
    auto it = std::lower_bound(vocab_.begin(), vocab_.end(), token, [](const std::string &a, std::string_view b) { return std::string_view(a) < b; });
    return (it != vocab_.end() && std::string_view(*it) == token) ? (uint32_t)(it - vocab_.begin()) : OI_NO_DOC;
  }
  // query text -> term ids (query_terms_of)
  std::vector<uint32_t> query_terms(std::string_view text) const {
    return query_terms_of(text, [&](std::string_view t) { return term_id(t); });
  }

 private:
  struct Raw { uint32_t term, doc, tf; };
  std::unordered_map<std::string, uint32_t> prov_;
  std::vector<std::string> terms_, vocab_, ids_;
  std::vector<Raw> raw_;
  std::vector<uint32_t> doc_len_, doc_ids_, tfs_;
  std::vector<uint64_t> term_off_;
  bool finished_ = false;
};

// The vocabulary of an index built from text on the device (oi_index_build_bm25_text): term t = bytes[offsets[t] ..
// offsets[t + 1]), ascending byte order.  Maps query text to term ids with IndexBuilder's rules.
class Vocabulary {
 public:
  uint32_t size() const { return offsets_.empty() ? 0 : (uint32_t)(offsets_.size() - 1); }
  std::string_view term(uint32_t t) const {
    return std::string_view(reinterpret_cast<const char *>(bytes_.data()) + offsets_.at(t), offsets_.at(t + 1) - offsets_[t]);
  }
  // term id of a token, or OI_NO_DOC when the token is not in the vocabulary
  uint32_t term_id(std::string_view token) const {
    uint32_t lo = 0, hi = size();
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (term(mid) < token) lo = mid + 1; else hi = mid;
    }
    return (lo < size() && term(lo) == token) ? lo : OI_NO_DOC;
  }
  std::vector<uint32_t> query_terms(std::string_view text) const {
    return query_terms_of(text, [&](std::string_view t) { return term_id(t); });
  }

 private:
  friend class GpuHybridSearch;
  std::vector<uint8_t> bytes_;
  std::vector<uint64_t> offsets_;
};

// ---- adapters over the C ABI ---------------------------------------------------------------------
class GpuHybridSearch final : public HybridSearch {
 public:
  // one shard on `device`; embeddings: n_docs x dim, L2-normalised, f32 (dtype F32) or bf16 bits (BF16)
  GpuHybridSearch(int device, uint32_t dim, uint32_t dtype, const void *embeddings, IndexBuilder &ix, uint32_t max_k = 100,
                  uint32_t max_batch = 64, uint32_t rrf_k = 60, float k1 = 1.2f, float b = 0.75f)
      : dim_(dim), rrf_k_(rrf_k) {
    ix.finish();
    open(device, ix.n_docs(), dim, dtype, embeddings, max_k, max_batch, [&] {
      ck(oi_index_load_bm25(h_, ix.term_offsets().data(), ix.doc_ids().data(), ix.tfs().data(), ix.doc_len().data(), ix.n_terms()));
    }, k1, b);
  }
  // the same index with its BM25 part built on the device from the posts' text: post i = texts[offsets[i] ..
  // offsets[i + 1]); `vocab` receives the vocabulary (what IndexBuilder::vocabulary() would hold)
  GpuHybridSearch(int device, uint32_t dim, uint32_t dtype, const void *embeddings, const uint8_t *texts, const uint64_t *offsets,
                  uint64_t n_posts, Vocabulary &vocab, uint32_t max_k = 100, uint32_t max_batch = 64, uint32_t rrf_k = 60,
                  float k1 = 1.2f, float b = 0.75f)
      : dim_(dim), rrf_k_(rrf_k) {
    open(device, n_posts, dim, dtype, embeddings, max_k, max_batch, [&] {
      uint32_t n_terms = 0;
      uint64_t n_bytes = 0;
      ck(oi_index_build_bm25_text(h_, texts, offsets, n_posts, &n_terms, &n_bytes));
      vocab.bytes_.resize(n_bytes);
      vocab.offsets_.resize((size_t)n_terms + 1);
      ck(oi_index_read_vocabulary(h_, vocab.bytes_.data(), vocab.offsets_.data()));
    }, k1, b);
  }
  ~GpuHybridSearch() override { oi_index_destroy(h_); }
  GpuHybridSearch(const GpuHybridSearch &) = delete;
  GpuHybridSearch &operator=(const GpuHybridSearch &) = delete;

  std::vector<std::vector<Hit>> search(const std::vector<SearchQuery> &queries, size_t k) const override {
    const uint32_t nq = (uint32_t)queries.size();
    std::vector<float> emb;
    std::vector<uint32_t> terms, offs{0};
    emb.reserve((size_t)nq * dim_);
    for (const SearchQuery &q : queries) {
      if (q.embedding.size() != dim_) throw DomainError::source_failure("gpu-search", "query embedding has the wrong dimension");
      emb.insert(emb.end(), q.embedding.begin(), q.embedding.end());
      terms.insert(terms.end(), q.terms.begin(), q.terms.end());
      offs.push_back((uint32_t)terms.size());
    }
    const size_t n = (size_t)nq * k;
    std::vector<uint32_t> ids(n), rc(n), rb(n);
    std::vector<float> rrf(n);
    if (terms.empty()) terms.push_back(0);  // a valid pointer for an all-empty batch
    ck(oi_search_hybrid(h_, emb.data(), terms.data(), offs.data(), nq, (uint32_t)k, rrf_k_, ids.data(), rrf.data(), rc.data(), rb.data()));
    std::vector<std::vector<Hit>> out(nq);
    for (uint32_t j = 0; j < nq; ++j)
      for (size_t i = 0; i < k; ++i) {
        const size_t at = (size_t)j * k + i;
        if (ids[at] == OI_NO_DOC) break;  // padding
        out[j].push_back(Hit{ids[at], rrf[at], rc[at], rb[at]});
      }
    return out;
  }
  oi_index *handle() const { return h_; }

 private:
  void ck(oi_status s) const {
    if (s != OI_OK) throw DomainError::source_failure("gpu-search", oi_last_error(h_));
  }
  // creates the index, loads the embeddings, runs `load_bm25` and finalizes; destroys the index on any failure
  template <class LoadBm25>
  void open(int device, uint64_t n_docs, uint32_t dim, uint32_t dtype, const void *embeddings, uint32_t max_k, uint32_t max_batch,
            LoadBm25 &&load_bm25, float k1, float b) {
    oi_index_desc d{};
    d.struct_size = sizeof(d);
    d.device = device; d.n_docs = n_docs; d.doc_base = 0; d.dim = dim; d.dtype = dtype; d.max_k = max_k; d.max_batch = max_batch;
    if (oi_index_create(&d, &h_) != OI_OK) throw DomainError::source_failure("gpu-search", oi_last_error(nullptr));
    try {
      ck(oi_index_load_embeddings(h_, embeddings, 0, n_docs));
      load_bm25();
      oi_bm25_params p{};
      p.struct_size = sizeof(p);
      p.k1 = k1; p.b = b; p.avgdl = 0.0f; p.n_docs_global = 0; p.global_df = nullptr;
      ck(oi_index_bm25_finalize(h_, &p));
    } catch (...) {
      oi_index_destroy(h_);
      throw;
    }
  }
  oi_index *h_ = nullptr;
  uint32_t dim_, rrf_k_;
};

// The reference's social summary (SpeculationEngine::social_summary, src/domain/engine/speculation_engine.rs:70-125).
struct SocialSummary {
  uint64_t total = 0, bullish = 0, bearish = 0, neutral = 0;
  double net_sentiment = 0.0, speculation_index = 0.0;
  double bull_bear_ratio = -1.0;  // -1: no bearish post (the reference's Option::None)
};

// ---- fusion signals on top of the summary: what SpeculationEngine::aggregate derives next (O(1) scalar arithmetic on
// the summary and a market snapshot; src/domain/engine/speculation_engine.rs:43-66).  Host code by design.
struct EngineConfig {  // src/domain/engine/config.rs:2-33, same names and defaults
  double bull_bear_threshold = 0.2, net_sentiment_threshold = 0.05, price_move_threshold = 1.0;
  double crowding_weight_spec = 0.5, crowding_weight_rvol = 0.3, crowding_weight_iv = 0.2, rvol_cap = 3.0;
  uint64_t min_sample = 10, confidence_low = 10, confidence_high = 50;
};
struct MarketSummary {  // the fields the fusion reads (speculation_engine.rs:127-148)
  double pct_change = 0.0;
  bool has_rvol = false;
  double rvol = 0.0;
  bool has_iv_rank = false;
  double iv_rank = 0.0;
  // a zero previous close gives pct_change 0, a zero average volume no rvol
  static MarketSummary from_snapshot(double last_price, double previous_close, uint64_t volume, uint64_t avg_volume) {
    MarketSummary m;
    m.pct_change = previous_close == 0.0 ? 0.0 : (last_price - previous_close) / previous_close * 100.0;
    m.has_rvol = avg_volume != 0;
    if (m.has_rvol) m.rvol = (double)volume / (double)avg_volume;
    return m;
  }
};
enum class Alignment { ConfirmingBullish = 0, ConfirmingBearish = 1, Diverging = 2, Quiet = 3 };
enum class Confidence { Low = 0, Medium = 1, High = 2 };

inline double clamp01(double x) { return x < 0.0 ? 0.0 : (x > 1.0 ? 1.0 : x); }
// weighted blend of the components that are present, renormalised over their weights (speculation_engine.rs:151-176)
inline double crowding(const SocialSummary &s, const MarketSummary *m, const EngineConfig &cfg = EngineConfig()) {
  double weighted = 0.0, weight_sum = 0.0;
  if (s.total > 0) { weighted += cfg.crowding_weight_spec * s.speculation_index; weight_sum += cfg.crowding_weight_spec; }
  if (m && m->has_rvol) { weighted += cfg.crowding_weight_rvol * clamp01(m->rvol / cfg.rvol_cap); weight_sum += cfg.crowding_weight_rvol; }
  if (m && m->has_iv_rank) { weighted += cfg.crowding_weight_iv * clamp01(m->iv_rank); weight_sum += cfg.crowding_weight_iv; }
  return weight_sum == 0.0 ? 0.0 : clamp01(weighted / weight_sum);
}
// does the crowd agree with the tape (speculation_engine.rs:178-208)
inline Alignment alignment(const SocialSummary &s, const MarketSummary *m, const EngineConfig &cfg = EngineConfig()) {
  if (!m || s.total < cfg.min_sample) return Alignment::Quiet;
  const double a = s.net_sentiment, p = m->pct_change;
  if (!(std::fabs(a) >= cfg.net_sentiment_threshold) || !(std::fabs(p) >= cfg.price_move_threshold)) return Alignment::Quiet;
  if (a > 0.0 && p > 0.0) return Alignment::ConfirmingBullish;
  if (!(a > 0.0) && !(p > 0.0)) return Alignment::ConfirmingBearish;
  return Alignment::Diverging;
}
// sample-size bucket; reversed thresholds are normalised first (src/domain/values/speculation.rs:29-42)
inline Confidence confidence(uint64_t n, uint64_t low, uint64_t high) {
  const uint64_t lo = std::min(low, high), hi = std::max(low, high);
  return n < lo ? Confidence::Low : (n < hi ? Confidence::Medium : Confidence::High);
}

// Replaces LexiconAnalyzer::analyze (src/adapters/analyzer/lexicon.rs:82-87) with the batched GPU scorer.  Owns an
// oi_lexicon handle: the stream and the device buffers are created once and reused by every call.
class GpuLexiconAnalyzer final : public PostAnalyzer {
 public:
  explicit GpuLexiconAnalyzer(int device = 0) {
    if (oi_lexicon_create(device, 1u << 20, 1u << 12, &lx_) != OI_OK) throw DomainError::source_failure("gpu-lexicon", oi_last_error(nullptr));
  }
  ~GpuLexiconAnalyzer() override { oi_lexicon_destroy(lx_); }
  GpuLexiconAnalyzer(const GpuLexiconAnalyzer &) = delete;
  GpuLexiconAnalyzer &operator=(const GpuLexiconAnalyzer &) = delete;

  std::vector<PostSignal> analyze(const std::vector<SocialPost> &posts) const override { return run(posts, nullptr); }
  // analyze + the batch's social summary in the same call (bull/bear threshold of EngineConfig::default: 0.2)
  std::vector<PostSignal> analyze(const std::vector<SocialPost> &posts, SocialSummary *summary, double threshold = 0.2) const {
    oi_social_summary s{};
    std::vector<PostSignal> out = run(posts, summary ? &s : nullptr, threshold);
    if (summary) {
      summary->total = s.total; summary->bullish = s.bullish; summary->bearish = s.bearish; summary->neutral = s.neutral;
      summary->net_sentiment = s.net_sentiment; summary->speculation_index = s.speculation_index; summary->bull_bear_ratio = s.bull_bear_ratio;
    }
    return out;
  }
  // packed form (texts already concatenated): what a caller with its own buffers uses; returns seconds spent in the call
  void run_packed(const uint8_t *blob, const uint64_t *offs, uint64_t n, double *pol, uint8_t *spec, oi_social_summary *summary = nullptr) const {
    if (oi_lexicon_run(lx_, blob, offs, n, pol, spec, nullptr, nullptr, 0.2, summary) != OI_OK)
      throw DomainError::source_failure("gpu-lexicon", oi_last_error(nullptr));
  }

 private:
  std::vector<PostSignal> run(const std::vector<SocialPost> &posts, oi_social_summary *summary, double threshold = 0.2) const {
    std::string blob;
    std::vector<uint64_t> offs{0};
    for (const SocialPost &p : posts) {
      blob += p.text;
      offs.push_back(blob.size());
    }
    const size_t n = posts.size();
    std::vector<double> pol(n);
    std::vector<uint8_t> spec(n);
    if (blob.empty()) blob.push_back('\0');
    if (oi_lexicon_run(lx_, reinterpret_cast<const uint8_t *>(blob.data()), offs.data(), n, pol.data(), spec.data(), nullptr, nullptr, threshold,
                       summary) != OI_OK)
      throw DomainError::source_failure("gpu-lexicon", oi_last_error(nullptr));
    std::vector<PostSignal> out(n);
    for (size_t i = 0; i < n; ++i) out[i] = PostSignal{pol[i], spec[i] != 0};
    if (out.size() != posts.size()) throw DomainError(DomainError::AnalyzerMismatch, "", "analyzer returned a different number of signals");
    return out;
  }
  oi_lexicon *lx_ = nullptr;
};

}  // namespace openintel
