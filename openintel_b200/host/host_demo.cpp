// host_demo.cpp — end-to-end use of the C++ host layer: posts + embeddings in, hybrid hits out.
//   host_demo <posts.txt> <embeddings.f32> <dim> <queries.txt> <query_embeddings.f32> <k>
// posts.txt / queries.txt: one text per line.  Prints one line per hit: "q rank doc_id rrf rc rb",
// then one line per post "signal i polarity speculative" from the GPU PostAnalyzer.
//   host_demo --store <posts.db> <queries.txt> <query_embeddings.f32> <k>
// lifts the index out of a SQLite post store (openintel_store.hpp) and prints "hit q rank doc_id rrf rc rb post_id".
//   host_demo --analyze <posts.db> [last_price previous_close volume avg_volume [iv_rank]]
// the reference's analyze use case over a store with the GPU PostAnalyzer injected (see analyze_mode).
//   host_demo --lexicon-bench <n_posts> [reps]
// GPU PostAnalyzer throughput without any Python in the loop: n_posts synthetic posts are packed once in C++, then
// `reps` calls of the handle API are timed (host buffers in, host buffers out); prints posts/s and text GB/s.
#include <chrono>
#include <cstdio>
#include <fstream>
#include <iostream>

#include "openintel_host.hpp"
#include "openintel_store.hpp"

using namespace openintel;

static std::vector<std::string> read_lines(const char *path) {
  std::ifstream f(path);
  std::vector<std::string> out;
  for (std::string line; std::getline(f, line);) out.push_back(line);
  return out;
}
static std::vector<float> read_f32(const char *path) {
  std::ifstream f(path, std::ios::binary | std::ios::ate);
  const std::streamsize n = f.tellg();
  f.seekg(0);
  std::vector<float> v((size_t)n / sizeof(float));
  f.read(reinterpret_cast<char *>(v.data()), n);
  return v;
}

static int store_mode(int argc, char **argv) {
  if (argc != 6) { std::fprintf(stderr, "usage: host_demo --store posts.db queries.txt qemb.f32 k\n"); return 2; }
  const SqlitePostStore store(argv[2]);
  const std::vector<std::string> qtexts = read_lines(argv[3]);
  std::vector<float> qemb = read_f32(argv[4]);
  const size_t k = std::stoul(argv[5]);
  const uint32_t dim = store.dim();
  if (qemb.size() != qtexts.size() * dim) throw std::runtime_error("query embedding file size mismatch");
  Vocabulary vocab;
  std::vector<std::string> post_ids;
  const auto search = lift_index(store, vocab, post_ids, 0, (uint32_t)k, (uint32_t)std::max<size_t>(qtexts.size(), 1));
  std::vector<SearchQuery> queries;
  for (size_t j = 0; j < qtexts.size(); ++j) {
    SearchQuery q;
    q.embedding.assign(qemb.begin() + j * dim, qemb.begin() + (j + 1) * dim);
    float ss = 0.0f;  // queries are normalised by the caller (SPEC §2)
    for (float v : q.embedding) ss += v * v;
    const float nrm = std::sqrt(ss);
    if (nrm > 0.0f)
      for (float &v : q.embedding) v /= nrm;
    q.terms = vocab.query_terms(qtexts[j]);
    queries.push_back(std::move(q));
  }
  const HybridSearch &port = *search;
  const auto hits = port.search(queries, k);
  for (size_t j = 0; j < hits.size(); ++j)
    for (size_t i = 0; i < hits[j].size(); ++i)
      std::printf("hit %zu %zu %u %.9g %u %u %s\n", j, i, hits[j][i].doc_id, hits[j][i].rrf, hits[j][i].rank_cosine, hits[j][i].rank_bm25,
                  post_ids[hits[j][i].doc_id].c_str());
  std::printf("store %llu posts dim %u terms %u\n", (unsigned long long)store.n_posts(), dim, vocab.size());
  return 0;
}

// host_demo --analyze <posts.db> [last_price previous_close volume avg_volume [iv_rank]]
// The reference's `analyze` use case (src/application/analyze.rs:16-73) over the posts of a store, with the GPU
// PostAnalyzer injected through the `PostAnalyzer` port: posts -> one device call (signals + social summary) -> fusion
// signals on the host -> one line "report total bullish bearish neutral net spec_index crowding alignment confidence".
static int analyze_mode(int argc, char **argv) {
  if (argc != 3 && argc != 7 && argc != 8) {
    std::fprintf(stderr, "usage: host_demo --analyze posts.db [last_price previous_close volume avg_volume [iv_rank]]\n");
    return 2;
  }
  const SqlitePostStore store(argv[2]);
  std::vector<SocialPost> posts;
  store.for_each_post([&](const SocialPost &p) { posts.push_back(p); });
  MarketSummary market;
  const bool has_market = argc >= 7;
  if (has_market) {
    market = MarketSummary::from_snapshot(std::stod(argv[3]), std::stod(argv[4]), std::stoull(argv[5]), std::stoull(argv[6]));
    if (argc == 8) { market.has_iv_rank = true; market.iv_rank = std::stod(argv[7]); }
  }
  if (posts.empty() && !has_market) throw DomainError::source_failure("analyze", "no data");  // DomainError::NoData
  const EngineConfig cfg;
  const GpuLexiconAnalyzer gpu(0);
  const PostAnalyzer &analyzer = gpu;  // the use case sees the port only (src/application/analyze.rs:62-63 de-hard-wired)
  (void)analyzer;
  SocialSummary sum;
  std::vector<PostSignal> signals;
  if (!posts.empty()) signals = gpu.analyze(posts, &sum, cfg.bull_bear_threshold);
  if (signals.size() != posts.size()) throw DomainError::source_failure("analyze", "analyzer mismatch");
  static const char *kAlign[] = {"ConfirmingBullish", "ConfirmingBearish", "Diverging", "Quiet"};
  static const char *kConf[] = {"Low", "Medium", "High"};
  std::printf("report %llu %llu %llu %llu %.17g %.17g %.17g %s %s\n", (unsigned long long)sum.total, (unsigned long long)sum.bullish,
              (unsigned long long)sum.bearish, (unsigned long long)sum.neutral, sum.net_sentiment, sum.speculation_index,
              crowding(sum, has_market ? &market : nullptr, cfg), kAlign[(int)alignment(sum, has_market ? &market : nullptr, cfg)],
              kConf[(int)confidence(sum.total, cfg.confidence_low, cfg.confidence_high)]);
  return 0;
}

static int lexicon_bench(int argc, char **argv) {
  if (argc < 3) { std::fprintf(stderr, "usage: host_demo --lexicon-bench n_posts [reps]\n"); return 2; }
  const size_t n = std::stoul(argv[2]);
  const int reps = argc > 3 ? std::stoi(argv[3]) : 10;
  static const char *kWords[] = {"AAPL", "to", "the", "moon", "calls", "puts", "0dte", "yolo", "dump", "rally", "bagholder", "earnings", "holding",
                                 "$TSLA,", "squeeze", "red", "green", "today", "market", "is", "up", "down", "a", "lot"};
  std::string blob;
  std::vector<uint64_t> offs{0};
  uint64_t x = 88172645463325252ull;
  for (size_t i = 0; i < n; ++i) {
    x ^= x << 13; x ^= x >> 7; x ^= x << 17;
    const int len = 8 + (int)(x % 40);  // ~28 words, ~150 bytes: a typical post
    for (int w = 0; w < len; ++w) {
      x ^= x << 13; x ^= x >> 7; x ^= x << 17;
      blob += kWords[x % (sizeof(kWords) / sizeof(kWords[0]))];
      blob += ' ';
    }
    offs.push_back(blob.size());
  }
  std::vector<double> pol(n);
  std::vector<uint8_t> spec(n);
  GpuLexiconAnalyzer an(0);
  oi_social_summary sum{};
  an.run_packed(reinterpret_cast<const uint8_t *>(blob.data()), offs.data(), n, pol.data(), spec.data(), &sum);  // warm-up, buffers grow
  const auto t0 = std::chrono::steady_clock::now();
  for (int r = 0; r < reps; ++r) an.run_packed(reinterpret_cast<const uint8_t *>(blob.data()), offs.data(), n, pol.data(), spec.data(), nullptr);
  const double s = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() / reps;
  // the same call with the fused social summary (a sequential f64 sum on the device: the reference's order)
  const auto t1 = std::chrono::steady_clock::now();
  for (int r = 0; r < reps; ++r) an.run_packed(reinterpret_cast<const uint8_t *>(blob.data()), offs.data(), n, pol.data(), spec.data(), &sum);
  const double s_sum = std::chrono::duration<double>(std::chrono::steady_clock::now() - t1).count() / reps;
  std::printf("lexicon-bench posts %zu with_summary_ms_per_call %.3f summary_extra_ms %.3f\n", n, s_sum * 1e3, (s_sum - s) * 1e3);
  std::printf("lexicon-bench posts %zu bytes %zu ms_per_call %.3f posts_per_s %.0f text_GBps %.3f bullish %llu bearish %llu neutral %llu net %.6f\n", n,
              blob.size(), s * 1e3, n / s, blob.size() / s / 1e9, (unsigned long long)sum.bullish, (unsigned long long)sum.bearish,
              (unsigned long long)sum.neutral, sum.net_sentiment);
  return 0;
}

int main(int argc, char **argv) {
  if (argc >= 2 && std::string(argv[1]) == "--lexicon-bench") {
    try {
      return lexicon_bench(argc, argv);
    } catch (const std::exception &e) {
      std::fprintf(stderr, "error: %s\n", e.what());
      return 1;
    }
  }
  if (argc >= 2 && std::string(argv[1]) == "--analyze") {
    try {
      return analyze_mode(argc, argv);
    } catch (const DomainError &e) {
      std::fprintf(stderr, "DomainError(%d): %s\n", (int)e.kind, e.what());
      return 1;
    } catch (const std::exception &e) {
      std::fprintf(stderr, "error: %s\n", e.what());
      return 1;
    }
  }
  if (argc >= 2 && std::string(argv[1]) == "--store") {
    try {
      return store_mode(argc, argv);
    } catch (const DomainError &e) {
      std::fprintf(stderr, "DomainError(%d): %s\n", (int)e.kind, e.what());
      return 1;
    } catch (const std::exception &e) {
      std::fprintf(stderr, "error: %s\n", e.what());
      return 1;
    }
  }
  if (argc != 7) { std::fprintf(stderr, "usage: host_demo posts.txt emb.f32 dim queries.txt qemb.f32 k\n"); return 2; }
  try {
    const std::vector<std::string> texts = read_lines(argv[1]);
    const std::vector<float> emb = read_f32(argv[2]);
    const uint32_t dim = (uint32_t)std::stoul(argv[3]);
    const std::vector<std::string> qtexts = read_lines(argv[4]);
    const std::vector<float> qemb = read_f32(argv[5]);
    const size_t k = std::stoul(argv[6]);
    if (emb.size() != texts.size() * dim || qemb.size() != qtexts.size() * dim) throw std::runtime_error("embedding file size mismatch");

    IndexBuilder ix;
    std::vector<SocialPost> posts;
    for (size_t i = 0; i < texts.size(); ++i) {
      SocialPost p;
      p.id = "post-" + std::to_string(i);
      p.source = "reddit";
      p.text = texts[i];
      posts.push_back(p);
      ix.add(p);
    }
    GpuHybridSearch search(0, dim, OI_DTYPE_F32, emb.data(), ix, (uint32_t)k, (uint32_t)std::max<size_t>(qtexts.size(), 1));
    std::vector<SearchQuery> queries;
    for (size_t j = 0; j < qtexts.size(); ++j) {
      SearchQuery q;
      q.embedding.assign(qemb.begin() + j * dim, qemb.begin() + (j + 1) * dim);
      q.terms = ix.query_terms(qtexts[j]);
      queries.push_back(std::move(q));
    }
    const HybridSearch &port = search;  // callers hold the port, not the adapter
    const auto hits = port.search(queries, k);
    for (size_t j = 0; j < hits.size(); ++j)
      for (size_t i = 0; i < hits[j].size(); ++i)
        std::printf("hit %zu %zu %u %.9g %u %u\n", j, i, hits[j][i].doc_id, hits[j][i].rrf, hits[j][i].rank_cosine, hits[j][i].rank_bm25);
    GpuLexiconAnalyzer analyzer(0);
    const PostAnalyzer &aport = analyzer;
    const auto sig = aport.analyze(posts);
    for (size_t i = 0; i < sig.size(); ++i) std::printf("signal %zu %.17g %d\n", i, sig[i].polarity, sig[i].speculative ? 1 : 0);
  } catch (const DomainError &e) {
    std::fprintf(stderr, "DomainError(%d): %s\n", (int)e.kind, e.what());
    return 1;
  } catch (const std::exception &e) {
    std::fprintf(stderr, "error: %s\n", e.what());
    return 1;
  }
  return 0;
}
