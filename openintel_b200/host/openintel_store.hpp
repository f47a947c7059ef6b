// openintel_store.hpp — the SQLite post store read from C++ and the index lift out of it
// (SURVEY.md §8 row a5 / §8(f) rank 1; BASELINE.json configs[0] "SQLite-backed").
//
// Same schema as openintel_b200/store.py (which creates and fills the store in the tests): table `posts` with the
// reference's SocialPost fields (src/domain/entities/social_post.rs:30-38) keyed by a dense `doc_id`, table
// `embeddings` with one little-endian f32 BLOB per post, `meta('dim')`.  The reference keeps no store (SURVEY.md §0).
//
// The image ships libsqlite3.so.0 but no sqlite3.h, so the dozen C entry points used here are declared by hand
// and bound with dlopen at run time; the SQLite C API is ABI-stable.  Header-only, CPU only: scoring stays in
// libopenintel_gpu.so.
#pragma once
#include <dlfcn.h>

#include <cmath>
#include <memory>

#include "openintel_host.hpp"

namespace openintel {

class SqlitePostStore {
 public:
  explicit SqlitePostStore(const std::string &path) {
    api_ = load_api();
    if (api_->open_v2(path.c_str(), &db_, 1 /* SQLITE_OPEN_READONLY */, nullptr) != 0) {
      const std::string msg = db_ ? api_->errmsg(db_) : "cannot open";
      if (db_) api_->close(db_);
      throw DomainError::source_failure("post-store", path + ": " + msg);
    }
    Stmt s(*this, "SELECT value FROM meta WHERE key = 'dim'");
    if (s.step()) dim_ = (uint32_t)std::stoul(s.text(0));
    Stmt c(*this, "SELECT COUNT(*) FROM posts");
    if (c.step()) n_posts_ = (uint64_t)c.i64(0);
  }
  ~SqlitePostStore() {
    if (db_) api_->close(db_);
  }
  SqlitePostStore(const SqlitePostStore &) = delete;
  SqlitePostStore &operator=(const SqlitePostStore &) = delete;

  uint32_t dim() const { return dim_; }  // 0 = the store holds no embeddings
  uint64_t n_posts() const { return n_posts_; }

  // every post in doc_id order; doc ids must be dense 0..N-1 (they are the index's u32 doc ids)
  template <class F>
  void for_each_post(F &&f) const {
    Stmt s(*this, "SELECT doc_id, id, source, author, text, engagement FROM posts ORDER BY doc_id");
    int64_t expect = 0;
    while (s.step()) {
      if (s.i64(0) != expect) throw DomainError::source_failure("post-store", "posts.doc_id must be dense 0..N-1 (gap at " + std::to_string(expect) + ")");
      ++expect;
      SocialPost p;
      p.id = s.text(1);
      p.source = s.text(2);
      p.author = s.text(3);
      p.text = s.text(4);
      p.engagement = (uint32_t)s.i64(5);
      f(p);
    }
  }

  // [n_posts][dim] f32, each row L2-normalised in f32 (SPEC §2: stored rows are normalised at build time; a zero
  // row stays zero); a post without an embedding is an error
  std::vector<float> embeddings() const {
    if (dim_ == 0) throw DomainError::source_failure("post-store", "store has no embeddings");
    std::vector<float> out((size_t)n_posts_ * dim_);
    Stmt s(*this, "SELECT doc_id, vec FROM embeddings ORDER BY doc_id");
    uint64_t got = 0;
    while (s.step()) {
      if ((uint64_t)s.i64(0) != got || got >= n_posts_) throw DomainError::source_failure("post-store", "embedding missing for doc " + std::to_string(got));
      if ((size_t)s.bytes(1) != (size_t)dim_ * 4) throw DomainError::source_failure("post-store", "doc " + std::to_string(got) + ": embedding has the wrong size");
      float *row = out.data() + (size_t)got * dim_;
      std::memcpy(row, s.blob(1), (size_t)dim_ * 4);
      float ss = 0.0f;
      for (uint32_t i = 0; i < dim_; ++i) ss += row[i] * row[i];
      const float nrm = std::sqrt(ss);
      if (nrm > 0.0f)
        for (uint32_t i = 0; i < dim_; ++i) row[i] /= nrm;
      ++got;
    }
    if (got != n_posts_) throw DomainError::source_failure("post-store", "embedding missing for doc " + std::to_string(got));
    return out;
  }

 private:
  struct Api {
    void *lib = nullptr;
    int (*open_v2)(const char *, void **, int, const char *) = nullptr;
    int (*close)(void *) = nullptr;
    int (*prepare_v2)(void *, const char *, int, void **, const char **) = nullptr;
    int (*step)(void *) = nullptr;
    int (*finalize)(void *) = nullptr;
    long long (*column_int64)(void *, int) = nullptr;
    const unsigned char *(*column_text)(void *, int) = nullptr;
    const void *(*column_blob)(void *, int) = nullptr;
    int (*column_bytes)(void *, int) = nullptr;
    const char *(*errmsg)(void *) = nullptr;
  };
  static const Api *load_api() {
    static Api api;
    static bool tried = false;
    if (!tried) {
      tried = true;
      for (const char *n : {"libsqlite3.so.0", "libsqlite3.so"}) {
        api.lib = dlopen(n, RTLD_NOW);
        if (api.lib) break;
      }
      if (api.lib) {
        auto sym = [&](const char *name) { return dlsym(api.lib, name); };
        api.open_v2 = (decltype(api.open_v2))sym("sqlite3_open_v2");
        api.close = (decltype(api.close))sym("sqlite3_close");
        api.prepare_v2 = (decltype(api.prepare_v2))sym("sqlite3_prepare_v2");
        api.step = (decltype(api.step))sym("sqlite3_step");
        api.finalize = (decltype(api.finalize))sym("sqlite3_finalize");
        api.column_int64 = (decltype(api.column_int64))sym("sqlite3_column_int64");
        api.column_text = (decltype(api.column_text))sym("sqlite3_column_text");
        api.column_blob = (decltype(api.column_blob))sym("sqlite3_column_blob");
        api.column_bytes = (decltype(api.column_bytes))sym("sqlite3_column_bytes");
        api.errmsg = (decltype(api.errmsg))sym("sqlite3_errmsg");
        if (!api.open_v2 || !api.close || !api.prepare_v2 || !api.step || !api.finalize || !api.column_int64 || !api.column_text ||
            !api.column_blob || !api.column_bytes || !api.errmsg)
          api.lib = nullptr;
      }
    }
    if (!api.lib) throw DomainError::source_failure("post-store", "libsqlite3.so.0 is not loadable");
    return &api;
  }
  // one prepared statement, finalised on scope exit
  struct Stmt {
    const SqlitePostStore &st;
    void *h = nullptr;
    Stmt(const SqlitePostStore &s, const char *sql) : st(s) {
      if (st.api_->prepare_v2(st.db_, sql, -1, &h, nullptr) != 0) throw DomainError::source_failure("post-store", st.api_->errmsg(st.db_));
    }
    ~Stmt() {
      if (h) st.api_->finalize(h);
    }
    bool step() {
      const int rc = st.api_->step(h);
      if (rc == 100) return true;   // SQLITE_ROW
      if (rc == 101) return false;  // SQLITE_DONE
      throw DomainError::source_failure("post-store", st.api_->errmsg(st.db_));
    }
    long long i64(int c) { return st.api_->column_int64(h, c); }
    std::string text(int c) {
      const unsigned char *p = st.api_->column_text(h, c);
      return p ? std::string(reinterpret_cast<const char *>(p), (size_t)st.api_->column_bytes(h, c)) : std::string();
    }
    const void *blob(int c) { return st.api_->column_blob(h, c); }
    int bytes(int c) { return st.api_->column_bytes(h, c); }
  };

  const Api *api_ = nullptr;
  void *db_ = nullptr;
  uint32_t dim_ = 0;
  uint64_t n_posts_ = 0;
};

// store -> GPU index: the posts' text goes to the device in one packed blob, where the vocabulary and the CSR are built
// (oi_index_build_bm25_text); the normalised embeddings are loaded next to them.  `vocab` maps query text to term ids
// (Vocabulary::query_terms) and `post_ids` doc ids back to post ids; both stay with the caller.
inline std::unique_ptr<GpuHybridSearch> lift_index(const SqlitePostStore &store, Vocabulary &vocab, std::vector<std::string> &post_ids,
                                                   int device = 0, uint32_t max_k = 100, uint32_t max_batch = 16,
                                                   std::vector<float> *rows_out = nullptr) {
  std::string blob;
  std::vector<uint64_t> offs{0};
  post_ids.clear();
  store.for_each_post([&](const SocialPost &p) {
    blob += p.text;
    offs.push_back(blob.size());
    post_ids.push_back(p.id);
  });
  if (blob.empty()) blob.push_back('\0');  // a valid pointer for a store without text
  std::vector<float> rows = store.embeddings();
  auto gs = std::make_unique<GpuHybridSearch>(device, store.dim(), (uint32_t)OI_DTYPE_F32, rows.data(),
                                              reinterpret_cast<const uint8_t *>(blob.data()), offs.data(), offs.size() - 1, vocab,
                                              max_k, max_batch);
  if (rows_out) *rows_out = std::move(rows);
  return gs;
}

}  // namespace openintel
