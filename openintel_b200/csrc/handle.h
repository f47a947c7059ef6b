// handle.h — the opaque oi_index: everything one shard owns on one GPU.
#pragma once
#include "internal.h"

struct OiBm25;  // bm25.cu
struct OiComm;  // comm.cu
struct OiGemm;  // cosine_gemm.cu

#define OI_PIN_BYTES (1u << 20)
#define OI_SLOTS 4

struct oi_index {
  oi_index_desc desc{};
  int num_sms = 0;
  cudaStream_t stream = nullptr;
  std::mutex mu;       // calls on one handle are serialised (SURVEY §8b threading)
  std::string err;     // last error message (read through oi_last_error, which copies it under the lock)
  uint64_t launches = 0;
  // Every search call uses the handle's single set of workspaces.  The mutex serialises the ENQUEUE; the work of two
  // calls enqueued on different streams (`_dev` calls on caller streams, host-buffer calls on `stream`) is ordered on
  // the device by an event recorded at the end of every call and waited for by the next call's stream.
  cudaEvent_t ev_last = nullptr;
  cudaStream_t last_stream = nullptr;
  bool has_last = false;
  // hybrid call: the BM25 leg can run on a second stream next to the cosine GEMM (see api.cu hybrid_enqueue)
  cudaStream_t stream2 = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int hybrid_overlap = 0;      // 0 = legs back to back on one stream; 1 = co-resident "lite" kernels (GEMM 96 KB ring + BM25 with
                               // overlap_bm25_warps warps per CTA on every SM); 2 = SM partition (full kernels, overlap_gemm_sms SMs to the GEMM)
  int overlap_bm25_warps = 10;
  int overlap_bm25_slots = 1;
  int overlap_gemm_sms = 74;

  // embeddings
  void *d_emb = nullptr;
  uint64_t emb_rows_loaded = 0;  // rows [0, emb_rows_loaded) hold data: chunks must arrive in order (or overwrite loaded rows)
  int cosine_variant = 1;  // 0 = direct loads, 1 = bulk-copy pipeline with dynamic tiles
  int cosine_multi_query = 2;  // calls with several queries scan the matrix once per group of 4 (rows <= 1536 B): 2 = on the
                               // bulk-copy pipeline where the group fits the registers (f32), 1 = direct loads, 0 = off

  // per-call workspaces (device)
  OiCosineWorkspace cws;
  size_t cws_slots = 0;
  float *d_queries = nullptr;     // [max_batch][dim]
  u64 *d_keys_cos = nullptr;      // [max_batch][max_k] global cosine lists
  u64 *d_keys_bm25 = nullptr;     // [max_batch][max_k] global BM25 lists
  u64 *d_keys_local = nullptr;    // 2 x [max_batch][max_k] shard-local lists before the all-gather
  u64 *d_gather = nullptr;        // [world] x 2 x [max_batch][max_k]
  uint32_t *d_out_u32 = nullptr;  // 3 x [max_batch][max_k]
  float *d_out_f32 = nullptr;     // [max_batch][max_k]
  // small host-buffer calls go through one pinned staging block each way: one H2D copy of (queries | terms |
  // offsets) and one D2H copy of (ids | scores | ranks) instead of 3 + 4 copies from / to pageable memory
  // ... and there are OI_SLOTS such blocks: a host-buffer call owns one from its enqueue until it has copied its results
  // out, and the handle's lock is only held for the ENQUEUE -- while one thread waits for its results another one
  // already packs and enqueues the next call behind it on the stream (the reference awaits one &self from many tasks:
  // src/application/analyze.rs:30-37).  The kernels of the calls still run one after the other (one set of workspaces).
  struct Slot {
    unsigned char *h_in = nullptr, *h_out = nullptr;  // OI_PIN_BYTES each (cudaHostAlloc)
    unsigned char *d_in = nullptr, *d_out = nullptr;  // device mirrors
    cudaEvent_t done = nullptr;                       // recorded behind the call's last copy
    bool busy = false;
  };
  Slot slots[4];
  std::condition_variable slot_cv;
  int no_pinned_staging = 0;  // tests: take the large-call path (direct copies from / to the caller's buffers)

  // batched cosine on the tensor cores (cosine_gemm.cu); workspace is created on first use
  OiGemm *gemm = nullptr;
  int gemm_min_batch = 4;      // batches of at least this many queries take the tcgen05 path (0 = never)
  int gemm_cap = 0;            // tests: candidate-list capacity override (0 = default)
  int gemm_force_2d = 0;       // tests: one 2-D TMA box per slab instead of the 3-D view
  int gemm_debug = 0;          // timing experiments only (see GemmParams::debug)
  int gemm_sample_tiles = 0;   // probe-pass tiles per CTA override (0 = default: 1/128 of the CTA's tiles); > 0 also forces the probe on small shards
  bool gemm_force_lite = false;  // experiments: always the 96 KB-ring kernel
  int gemm_pair = 1;           // 1: an even number of query tiles runs as CTA pairs (tcgen05.mma.cta_group::2, M = 256): 10 % faster
                               // than two independent M = 128 CTAs (profiles/r02_gemm_ab.md); 0 = never
  int gemm_pair_ring = 48;     // slabs (4 KB) in a pair CTA's ring at dim 768: 24 (96 KB) or 48 (192 KB)

  // BM25
  OiBm25 *bm25 = nullptr;
  int bm25_variant = 0;
  int bm25_warps = 0;         // tuning: warps per CTA (0 = default)
  int bm25_block_docs = 0;    // tuning: documents per block, a power of two >= 1024 (0 = default)
  int bm25_dense_div = 0;     // tuning (before finalize): a term in >= n_docs / div documents gets a dense column (0 = default 16)
  int bm25_items_per_warp = 0; // tuning: work items per warp the super-range count aims for (0 = default 16)
  int bm25_no_cold_bound = 0;  // tests: disable the cold-start bound (group maxima) of the selection pass
  int bm25_stage_slots = -1;  // tuning: staged 64-posting chunks per warp (-1 = default, 0 = none)
  // vocabulary of a BM25 part built from text (text_index.cu): term t = d_vocab[d_vocab_off[t] .. d_vocab_off[t + 1]);
  // NULL when the BM25 part came from a CSR.  Freed with the BM25 part (oi_bm25_free).
  uint8_t *d_vocab = nullptr;
  u64 *d_vocab_off = nullptr;
  uint64_t vocab_bytes = 0;

  // per-post lexicon signals (mention.cu), independent of the BM25 part: polarity f64 and speculative | source << 1
  // per post, [n_docs] each.  d_mention_io: grow-on-demand buffers of the calls too large for a pinned slot.
  double *d_sig_pol = nullptr;
  uint8_t *d_sig_flags = nullptr;
  bool has_signals = false;
  unsigned char *d_mention_io = nullptr;
  size_t mention_io_bytes = 0;
  // per-post creation times (seconds since the Unix epoch, [n_docs]) for the timelines, independent of the BM25 part
  // and of the signals; d_timeline_ws: the grow-on-demand keys / sort / segment workspace of the timeline call, and the
  // post mask and selection workspace of the co-mention calls
  int64_t *d_times = nullptr;
  bool has_times = false;
  unsigned char *d_timeline_ws = nullptr;
  size_t timeline_ws_bytes = 0;
  // per-post author ids and engagement ([n_docs] each) for the author runs, independent of the rest; n_authors = the
  // largest id + 1 (at least 1): the author part of the (term, author) keys
  uint32_t *d_author = nullptr, *d_engagement = nullptr;
  u64 n_authors = 0;
  bool has_authors = false;

  // multi-GPU
  OiComm *comm = nullptr;
  int rank = 0, world = 1;
  int comm_skip = 0;  // timing experiments only: skip the all-gather (results are then shard-local garbage)
  int comm_exchange = 0;  // 0 = ncclAllGather, 1 = peer-to-peer push over mapped buffers (set by oi_index_p2p_attach)

  uint32_t esize() const { return desc.dtype == OI_DTYPE_F32 ? 4u : 2u; }
  oi_status fail(oi_status code, const char *fmt, ...) __attribute__((format(printf, 3, 4)));
};

// api.cu: device-side ordering of the calls of one handle (see ev_last)
cudaError_t call_begin(oi_index *h, cudaStream_t st);
cudaError_t call_end(oi_index *h, cudaStream_t st);

// a failed CUDA call fails the handle's call (`h` in scope): out of memory for a failed allocation, a CUDA error else
#define OI_CK(call)                                                                              \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return h->fail(e_ == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA,       \
                     "%s failed: %s", #call, cudaGetErrorString(e_));                            \
  } while (0)

// blocks of `threads` for a grid-stride loop over n items: one per `threads` items, at most 16 per SM, at least 1
inline unsigned oi_grid(u64 n, int threads, int num_sms) {
  u64 b = (n + threads - 1) / threads;
  const u64 cap = (u64)num_sms * 16;
  if (b > cap) b = cap;
  return (unsigned)(b ? b : 1);
}

// A staging slot for one small host-buffer call.  Taken under the handle's lock (waiting, lock released, while all are
// busy); given back by the guard after the caller has copied its results out -- or on any early return.
struct SlotLease {
  oi_index *h;
  std::unique_lock<std::mutex> &lock;
  oi_index::Slot *sl;
  SlotLease(oi_index *h_, std::unique_lock<std::mutex> &lock_) : h(h_), lock(lock_), sl(nullptr) {
    for (;;) {
      for (oi_index::Slot &c : h->slots)
        if (!c.busy) { sl = &c; break; }
      if (sl) break;
      h->slot_cv.wait(lock);
    }
    sl->busy = true;
  }
  ~SlotLease() {
    if (!lock.owns_lock()) lock.lock();
    sl->busy = false;
    h->slot_cv.notify_one();
  }
  // the enqueue is complete: record the slot's event, let the next caller in, wait for this call's results
  oi_status finish(cudaStream_t st) {
    cudaError_t e = cudaEventRecord(sl->done, st);
    if (e == cudaSuccess) e = call_end(h, st);
    if (e == cudaSuccess) {
      lock.unlock();
      e = cudaEventSynchronize(sl->done);
      if (e != cudaSuccess) lock.lock();
    }
    if (e != cudaSuccess) return h->fail(OI_ERR_CUDA, "host-buffer call failed: %s", cudaGetErrorString(e));
    return OI_OK;
  }
};

// mention.cu
void oi_mention_free(oi_index *h);
// bm25.cu
void oi_bm25_free(oi_index *h);
// installs a CSR that already lives on the device (text_index.cu) as the BM25 part, as oi_index_load_bm25 leaves it;
// the arrays become the index's.  On failure they are freed and the index has no BM25 part.
oi_status oi_bm25_adopt(oi_index *h, uint32_t n_terms, uint64_t n_postings, u64 *d_term_off, uint32_t *d_doc_ids,
                        uint32_t *d_tfs, uint32_t *d_doc_len);
uint32_t oi_bm25_n_terms(const oi_index *h);  // 0 = no BM25 part
const u64 *oi_bm25_term_offsets(const oi_index *h);  // device term_offsets[n_terms + 1]; NULL = no BM25 part
const uint32_t *oi_bm25_doc_ids(const oi_index *h);  // device doc_ids[n_postings] (kept after finalize); NULL = no BM25 part
uint64_t oi_bm25_n_postings(const oi_index *h);  // 0 = no BM25 part or no posting
bool oi_bm25_finalized(const oi_index *h);
// re-indexes the BM25 part to n_terms terms over the same postings (text_index.cu's vocabulary union): d_term_off
// [n_terms + 1] on the device becomes the index's, the old offsets are freed.  Before finalize only.
void oi_bm25_replace_terms(oi_index *h, uint32_t n_terms, u64 *d_term_off);
uint32_t *oi_bm25_stage_terms(oi_index *h);  // device staging for the host call's flat term array
uint32_t *oi_bm25_stage_offs(oi_index *h);
// prep -> blocked scoring -> merge: shard-local sorted key lists d_out_keys[nq][k] (global doc ids)
// overlap: 0 = the stand-alone schedule (one CTA per SM, 20 warps); 1 = the "lite" schedule that shares every SM with a
// GEMM CTA (h->overlap_bm25_warps warps, 128 registers); 2 = full CTAs on the SMs the GEMM leaves free
oi_status oi_bm25_local_keys(oi_index *h, const uint32_t *d_q_terms, const uint32_t *d_q_offs, uint32_t nq,
                             uint32_t k, u64 *d_out_keys, cudaStream_t st, int overlap = 0);
size_t oi_bm25_stage_capacity(const oi_index *h);  // u32 slots of the flat term staging array
// cosine_gemm.cu
void oi_gemm_free(oi_index *h);
bool oi_gemm_eligible(const oi_index *h, uint32_t nq, uint32_t k);
// shard-local sorted key lists d_out_keys[nq][k] of nq f32 device queries; d_dump (tests) receives the
// raw nq x n_docs score matrix when not NULL
// lite: the 96 KB-ring kernel (co-resident with a BM25 CTA); max_ctas: 0 = every SM, else an upper bound of the grid
bool oi_gemm_lite_ok(const oi_index *h);
oi_status oi_gemm_local_keys(oi_index *h, const float *d_queries, uint32_t nq, uint32_t k, u64 *d_out_keys, float *d_dump,
                             cudaStream_t st, bool lite = false, uint32_t max_ctas = 0);
// comm.cu
void oi_comm_destroy(oi_index *h);
// all-gathers each rank's [nq][k] local lists and merges them into d_out [nq][k] on every rank
oi_status oi_comm_gather_merge(oi_index *h, const u64 *d_local, uint32_t nq, uint32_t k, u64 *d_out, cudaStream_t st);
// hybrid: d_local2 = [cosine nq x k | BM25 nq x k]; one all-gather, two merges
oi_status oi_comm_gather_merge2(oi_index *h, const u64 *d_local2, uint32_t nq, uint32_t k, u64 *d_out_cos, u64 *d_out_bm25, cudaStream_t st);
