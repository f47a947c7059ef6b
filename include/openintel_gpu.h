/* openintel_gpu.h — C ABI of libopenintel_gpu.so, the B200 (sm_100a) hybrid-retrieval engine.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference (Kloudy-Sky/openintel, Rust) has
 * no FFI and no search port of any kind (SURVEY.md §0), so there is no reference interface to
 * replace one-for-one; every entry point below cites the reference *convention* it is shaped
 * by, and INTEGRATION.md shows the Rust binding (`extern "C"` block + adapter implementing a
 * `HybridSearch` port in the style of src/domain/ports/post_analyzer.rs:7-11) a maintainer
 * would add.
 *
 * Conventions
 *  - plain pointers and sizes only; all `const T*` inputs and `T*` outputs of the non-`_dev`
 *    calls are caller-owned HOST memory (a Rust slice / Vec), borrowed for the call only —
 *    mirrors "borrowed slices in, owned Vec out" of the reference's ports
 *    (src/domain/ports/post_analyzer.rs:10).
 *  - every call returns an oi_status; 0 = ok.  No exception or panic crosses the boundary.
 *    The message for the last failure is oi_last_error(h) — the adapter maps it to
 *    DomainError::SourceFailure{name:"gpu-search", message} (src/domain/error.rs:17-18).
 *  - calls on one handle may come from many threads at once (the reference awaits ports
 *    concurrently on one &self: src/application/analyze.rs:30-37); the library serialises
 *    them internally (one set of workspaces per handle).  Host-buffer calls are blocking.
 *    `_dev` calls return after enqueueing; calls enqueued on DIFFERENT streams are ordered on
 *    the device by the library (an event recorded at the end of every call is waited for by
 *    the next call's stream), so they never overlap on the shared workspaces.
 *  - oi_last_error returns a pointer into thread-local storage: valid until the calling
 *    thread's next oi_last_error call.
 *  - result lists are ordered score-descending, ties by ascending doc id (docs/SPEC.md §1);
 *    short lists are padded with (OI_NO_DOC, 0).  Doc ids are GLOBAL (doc_base + local row).
 *  - there is no CPU fallback: without a CUDA device every call fails with OI_ERR_NO_DEVICE.
 */
#ifndef OPENINTEL_GPU_H
#define OPENINTEL_GPU_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OI_NO_DOC 0xFFFFFFFFu
#define OI_MAX_K 1024u
#define OI_UNIQUE_ID_BYTES 128
#define OI_P2P_HANDLE_BYTES 64

typedef int32_t oi_status;
enum {
  OI_OK = 0,
  OI_ERR_INVALID_ARG = 1,
  OI_ERR_NO_DEVICE = 2,
  OI_ERR_CUDA = 3,
  OI_ERR_OUT_OF_MEMORY = 4,
  OI_ERR_STATE = 5,       /* call made before the data it needs was loaded */
  OI_ERR_COMM = 6,        /* NCCL failure / NCCL not loadable */
  OI_ERR_UNSUPPORTED = 7
};

enum { OI_DTYPE_F32 = 0, OI_DTYPE_BF16 = 1 };

typedef struct oi_index oi_index; /* opaque; owns all device memory of one shard on one GPU */

typedef struct {
  uint32_t struct_size; /* = sizeof(oi_index_desc), for ABI evolution */
  int32_t device;       /* CUDA device ordinal */
  uint64_t n_docs;      /* documents held by THIS shard */
  uint64_t doc_base;    /* global id of this shard's first document (SPEC §5) */
  uint32_t dim;         /* embedding dimension; dim*sizeof(dtype) must be a multiple of 16 */
  uint32_t dtype;       /* OI_DTYPE_F32 | OI_DTYPE_BF16: storage type of the embedding matrix */
  uint32_t max_k;       /* largest k any search call will ask for (<= OI_MAX_K) */
  uint32_t max_batch;   /* largest number of queries per search call */
} oi_index_desc;

typedef struct {
  uint32_t struct_size;
  float k1;                  /* 1.2 */
  float b;                   /* 0.75 */
  float avgdl;               /* GLOBAL average doc length; <= 0 -> computed from this shard */
  uint64_t n_docs_global;    /* GLOBAL corpus size N for idf; 0 -> this shard's n_docs */
  const uint32_t *global_df; /* GLOBAL df per term [n_terms]; NULL -> this shard's list lengths */
} oi_bm25_params;

/* ---- lifecycle (adapter construction at the composition roots, src/main.rs:16-47) -------- */
oi_status oi_index_create(const oi_index_desc *desc, oi_index **out);
void oi_index_destroy(oi_index *h);
/* never NULL; h == NULL returns the calling thread's last creation error */
const char *oi_last_error(const oi_index *h);
/* library / build identification, e.g. "openintel_gpu 0.1 sm_100a" */
const char *oi_version(void);

/* ---- embeddings ---------------------------------------------------------------------------- */
/* rows [first_doc, first_doc+n) (shard-local numbering), already L2-normalised, in the index dtype.  Chunks must
 * extend the loaded prefix or rewrite rows inside it (first_doc <= rows loaded so far): searches are refused until
 * every row has been loaded, so uninitialised memory is never scored. */
oi_status oi_index_load_embeddings(oi_index *h, const void *rows, uint64_t first_doc, uint64_t n);
/* generate this shard's rows on the device (SPEC §9, stream 0, rows doc_base..doc_base+n_docs) */
oi_status oi_index_synth_embeddings(oi_index *h, uint64_t seed);
/* copy rows back to the host (tests / index export) */
oi_status oi_index_read_embeddings(oi_index *h, void *rows, uint64_t first_doc, uint64_t n);

/* ---- BM25 inverted index (SPEC §3) --------------------------------------------------------- */
/* shard-local CSR: term_offsets[n_terms+1], doc_ids/tfs[term_offsets[n_terms]] (doc ids local,
 * ascending inside a list), doc_len[n_docs].  Must be followed by oi_index_bm25_finalize.
 * The offsets are checked on the host, the postings on the device after the copy (doc ids inside the
 * shard, strictly ascending per list): a malformed CSR is OI_ERR_INVALID_ARG naming the first bad
 * posting, and leaves the index without a BM25 part. */
oi_status oi_index_load_bm25(oi_index *h, const uint64_t *term_offsets, const uint32_t *doc_ids,
                             const uint32_t *tfs, const uint32_t *doc_len, uint32_t n_terms);
/* build the synthetic shard-local CSR on the device (SPEC §9); zipf_cdf[vocab] from the host */
oi_status oi_index_synth_bm25(oi_index *h, uint64_t seed, uint32_t vocab, const double *zipf_cdf);
/* posts -> this shard's BM25 part, on the device: post i = texts[offsets[i] .. offsets[i+1]) (host memory),
 * n_posts == the shard's n_docs, doc ids local in input order.  Tokenizer = SPEC §6; vocabulary = the distinct tokens
 * in ascending byte order, term id = rank in it; doc_len = token count; tf = occurrences of the term in the post
 * (SPEC §3).  Leaves the index exactly as oi_index_load_bm25 with the host IndexBuilder's CSR would: follow with
 * oi_index_bm25_finalize.  out_n_terms / out_vocab_bytes size the buffers of oi_index_read_vocabulary.  A corpus
 * without any token is OI_ERR_INVALID_ARG (an index needs a term).  Any failure leaves the index without a BM25 part. */
oi_status oi_index_build_bm25_text(oi_index *h, const uint8_t *texts, const uint64_t *offsets, uint64_t n_posts,
                                   uint32_t *out_n_terms, uint64_t *out_vocab_bytes);
/* document-sharded index (SPEC §5), after oi_index_build_bm25_text, before oi_index_bm25_finalize: entry i =
 * terms[offsets[i] .. offsets[i+1]) (host memory), the concatenated vocabularies of all shards in any order, duplicates
 * allowed (the host gathers them over any transport).  The vocabulary becomes the sorted distinct union of the entries
 * (ascending byte order, a proper prefix first); this shard's CSR is re-indexed to it: term id = rank in the union,
 * terms this shard does not hold get empty lists, doc_ids / tfs / doc_len unchanged.  out_n_terms / out_vocab_bytes
 * size oi_index_read_vocabulary's buffers.  OI_ERR_STATE: the BM25 part was not built from text, or is finalized.
 * OI_ERR_INVALID_ARG: NULL pointers, no entries or more than 2^32 - 2, decreasing offsets, an entry that is empty or
 * holds a byte outside [0-9a-z] (tokens hold nothing else), a term of this shard missing from the entries.  A failed
 * call leaves the BM25 part and its vocabulary as they were; calling again with the same entries changes nothing. */
oi_status oi_index_bm25_union_vocabulary(oi_index *h, const uint8_t *terms, const uint64_t *offsets, uint64_t n_entries,
                                         uint32_t *out_n_terms, uint64_t *out_vocab_bytes);
/* the vocabulary of the BM25 part built from text (after oi_index_bm25_union_vocabulary: the union): term t =
 * bytes[offsets[t] .. offsets[t+1]), offsets[n_terms+1].  OI_ERR_STATE when the BM25 part did not come from text. */
oi_status oi_index_read_vocabulary(oi_index *h, uint8_t *bytes, uint64_t *offsets);
/* this shard's df per term and sum of doc lengths, to be summed over shards by the host */
oi_status oi_index_bm25_local_stats(oi_index *h, uint32_t *df_out, uint64_t *sum_doc_len,
                                    uint64_t *n_postings);
/* folds tf, doc length and the GLOBAL idf into per-posting weights; enables BM25 search */
oi_status oi_index_bm25_finalize(oi_index *h, const oi_bm25_params *params);
/* read the device-side CSR / weights back (tests): any pointer may be NULL */
oi_status oi_index_read_bm25(oi_index *h, uint64_t *term_offsets, uint32_t *doc_ids, uint32_t *tfs,
                             uint32_t *doc_len, float *weights);

/* ---- multi-GPU (SPEC §5): one process per GPU, all-gather of local top-k over NCCL ------- */
/* rank 0 creates the id, the host distributes it (any transport), every rank calls comm_init */
oi_status oi_comm_unique_id(uint8_t out[OI_UNIQUE_ID_BYTES]);
oi_status oi_index_comm_init(oi_index *h, int32_t rank, int32_t world_size,
                             const uint8_t unique_id[OI_UNIQUE_ID_BYTES]);

/* Optional peer-to-peer exchange (after oi_index_comm_init, all ranks on one NVLink box): instead of the all-gather,
 * every rank pushes its local lists straight into the other ranks' exchange buffers (CUDA IPC mappings, one kernel of
 * plain stores + an epoch flag per peer) and merges as soon as all flags have arrived.  Every rank exports the handle
 * of its buffer, the host distributes the `world_size` handles (any transport), every rank attaches; from then on the
 * sharded search calls use the push ("comm_exchange" option: 1 = push, 0 = back to ncclAllGather).  Results are
 * identical.  oi_index_p2p_status reports the number of exchanges and whether any wait for a peer timed out. */
oi_status oi_index_p2p_export(oi_index *h, uint8_t out[OI_P2P_HANDLE_BYTES]);
oi_status oi_index_p2p_attach(oi_index *h, const uint8_t *handles /* [world_size][OI_P2P_HANDLE_BYTES] */);
oi_status oi_index_p2p_status(oi_index *h, uint64_t *batches, uint32_t *timed_out);

/* ---- search: host buffers in, host buffers out (the calls the Rust adapter binds) --------- */
/* queries: nq x dim f32, L2-normalised.  out_ids/out_scores: nq x k. */
oi_status oi_search_cosine(oi_index *h, const float *queries, uint32_t nq, uint32_t k,
                           uint32_t *out_ids, float *out_scores);
/* query j's term ids are q_terms[q_offsets[j] .. q_offsets[j+1]): any number of raw ids; duplicates and unknown ids are
 * dropped and at most the first 64 distinct known terms (first-seen order) are scored (docs/SPEC.md §3).  One call may
 * carry at most 64 x max_batch ids in total. */
oi_status oi_search_bm25(oi_index *h, const uint32_t *q_terms, const uint32_t *q_offsets,
                         uint32_t nq, uint32_t k, uint32_t *out_ids, float *out_scores);
/* RRF (SPEC §4) of the two global top-k lists; out_rank_* are 1-based, 0 = not in that list */
oi_status oi_search_hybrid(oi_index *h, const float *queries, const uint32_t *q_terms,
                           const uint32_t *q_offsets, uint32_t nq, uint32_t k, uint32_t rrf_k,
                           uint32_t *out_ids, float *out_rrf, uint32_t *out_rank_cos,
                           uint32_t *out_rank_bm25);

/* ---- search, device-resident variants: every pointer is DEVICE memory on the index's GPU,
 * work is enqueued on `cuda_stream` (a cudaStream_t; NULL = the legacy default stream) and the
 * call returns without synchronising.  Used when inputs already live in HBM (bench `value`). */
oi_status oi_search_cosine_dev(oi_index *h, const float *d_queries, uint32_t nq, uint32_t k,
                               uint32_t *d_out_ids, float *d_out_scores, void *cuda_stream);
oi_status oi_search_bm25_dev(oi_index *h, const uint32_t *d_q_terms, const uint32_t *d_q_offsets,
                             uint32_t nq, uint32_t k, uint32_t *d_out_ids, float *d_out_scores,
                             void *cuda_stream);
oi_status oi_search_hybrid_dev(oi_index *h, const float *d_queries, const uint32_t *d_q_terms,
                               const uint32_t *d_q_offsets, uint32_t nq, uint32_t k, uint32_t rrf_k,
                               uint32_t *d_out_ids, float *d_out_rrf, uint32_t *d_out_rank_cos,
                               uint32_t *d_out_rank_bm25, void *cuda_stream);

/* ---- batched lexicon scorer: the GPU PostAnalyzer (SPEC §8; replaces LexiconAnalyzer::analyze,
 * src/adapters/analyzer/lexicon.rs:82-87; one output per input post, aligned to input order).
 * texts = concatenated UTF-8 bytes, post i = texts[offsets[i] .. offsets[i+1]).
 *
 * Handle form: the stream and the device buffers are created once (they grow on demand) and reused by every call; calls
 * on one handle are serialised.  oi_lexicon_run can also return the reference's social summary of the batch
 * (SpeculationEngine::social_summary, src/domain/engine/speculation_engine.rs:70-125: counts by the bull/bear threshold
 * -- 0.2 in EngineConfig::default, src/domain/engine/config.rs:18-33 --, mean polarity summed in input order,
 * speculation index, bull/bear ratio with -1 standing for "no bearish post"); out_summary may be NULL. */
typedef struct oi_lexicon oi_lexicon;
typedef struct {
  uint64_t total, bullish, bearish, neutral;
  double net_sentiment, speculation_index, bull_bear_ratio;
} oi_social_summary;
oi_status oi_lexicon_create(int32_t device, uint64_t reserve_bytes, uint64_t reserve_posts, oi_lexicon **out);
void oi_lexicon_destroy(oi_lexicon *lx);
oi_status oi_lexicon_run(oi_lexicon *lx, const uint8_t *texts, const uint64_t *offsets, uint64_t n_posts,
                         double *out_polarity, uint8_t *out_speculative, uint32_t *out_bull_hits,
                         uint32_t *out_bear_hits, double bull_bear_threshold, oi_social_summary *out_summary);
uint64_t oi_lexicon_launch_count(const oi_lexicon *lx);
/* convenience form on a per-device handle the library keeps for the life of the process */
oi_status oi_lexicon_analyze(int32_t device, const uint8_t *texts, const uint64_t *offsets,
                             uint64_t n_posts, double *out_polarity, uint8_t *out_speculative,
                             uint32_t *out_bull_hits, uint32_t *out_bear_hits);

/* ---- per-term social summaries over the BM25 posting lists (docs/SPEC.md §8a) ---------------
 * A post mentions term t iff one of its tokens equals t, so the posts that mention t are t's posting list, in doc
 * order.  With per-post lexicon signals loaded next to the BM25 part, one call returns the social summary of
 * oi_lexicon_run (same counts, same sequential f64 mean, same clamps) over each requested term's list.
 *
 * Document-sharded index: the mean is a SEQUENTIAL sum in doc order, so the shards run as a relay in rank order -- rank 0
 * calls with carry_in = NULL, rank r > 0 continues from the out_state of rank r - 1 -- and the last rank's out_summary is
 * bit-identical to the unsharded one.  (An all-reduce of per-shard partial sums would round differently.) */
#define OI_N_SOURCES 2 /* post sources in store-schema order: 0 = reddit, 1 = bluesky */

/* the running state of one term's summary after some prefix of the doc order */
typedef struct {
  uint64_t total, bullish, bearish, neutral, speculative; /* posts counted, by the bull/bear threshold, speculative */
  uint64_t by_source[OI_N_SOURCES];                       /* posts counted per source code */
  double sum; /* sequential f64 sum of the polarities so far, doc order (SPEC §8a) */
} oi_mention_state;

/* per-post lexicon signals of THIS shard, n = n_docs, host memory: polarity f64 (finite, in [-1, 1]; -0.0 is stored as
 * +0.0, which changes no sum), speculative 0/1, source < OI_N_SOURCES.  Checked before anything is replaced: a refused
 * call (OI_ERR_INVALID_ARG naming the first bad post) keeps the previous signals.  Independent of the BM25 part (a
 * rebuilt BM25 part keeps them). */
oi_status oi_index_load_post_signals(oi_index *h, const double *polarity, const uint8_t *speculative,
                                     const uint8_t *source);

/* for each of terms[0 .. n_terms): the social summary of the posts of this shard that mention the term
 * (its posting list), continued from carry_in[i] (NULL = nothing before this shard).  source: -1 = all
 * posts, else only that source's.  out_state[i] = the running state after this shard (may be NULL);
 * out_summary[i] = the summary of every post counted in out_state[i].  On the last shard of a relay,
 * that is the global summary.  Duplicate term ids are allowed (each gets its own output).
 * OI_ERR_STATE: no BM25 part, or no signals loaded.  OI_ERR_INVALID_ARG: NULL terms / out_summary, a term id >= the
 * BM25 part's n_terms, source outside -1 .. OI_N_SOURCES - 1.  Blocking; reads the posting lists only, so it works
 * before and after oi_index_bm25_finalize and changes neither. */
oi_status oi_index_mention_summary(oi_index *h, const uint32_t *terms, uint32_t n_terms, int32_t source,
                                   double bull_bear_threshold, const oi_mention_state *carry_in,
                                   oi_mention_state *out_state, oi_social_summary *out_summary);

/* ---- per-term timelines: the summaries above split by creation time (docs/SPEC.md §8b) ------
 * Bucket b of edges[0 .. n_buckets] is [edges[b], edges[b+1]) in seconds since the Unix epoch; a post outside
 * [edges[0], edges[n_buckets]) is in no bucket.  The summary of (term, bucket) is the §8a summary of the posts that
 * mention the term and fall in the bucket, in doc order, so with one bucket around all posts it equals
 * oi_index_mention_summary bit for bit.  A document-sharded index relays each (term, bucket) state in rank order
 * exactly as oi_index_mention_summary does. */

/* per-post creation times of THIS shard, n = n_docs, host memory, seconds since the Unix epoch (SPEC §8b).
 * Independent of the BM25 part and of the signals; a rebuilt BM25 part keeps them. */
oi_status oi_index_load_post_times(oi_index *h, const int64_t *created_at);

/* for term i of terms[0..n_terms) and bucket b of edges[0..n_buckets]: the social summary of this shard's posts that
 * mention the term and were created in [edges[b], edges[b+1]), doc order, continued from carry_in[i * n_buckets + b]
 * (NULL = nothing before this shard).  out_state (may be NULL) / out_summary: [n_terms][n_buckets], term-major.
 * source and duplicate term ids as in oi_index_mention_summary.  n_terms == 0 is a no-op.
 * OI_ERR_STATE: no BM25 part, no signals or no times loaded.  OI_ERR_INVALID_ARG: NULL terms / edges / out_summary,
 * n_buckets == 0, n_terms x n_buckets > 2^32 - 1 (the (term, bucket) keys are 32-bit), edges not strictly increasing,
 * a term id >= the BM25 part's n_terms, source outside -1 .. OI_N_SOURCES - 1.  A refused call changes nothing.
 * Blocking; reads the posting lists only, so it works before and after oi_index_bm25_finalize. */
oi_status oi_index_mention_timeline(oi_index *h, const uint32_t *terms, uint32_t n_terms, const int64_t *edges,
                                    uint32_t n_buckets, int32_t source, double bull_bear_threshold,
                                    const oi_mention_state *carry_in, oi_mention_state *out_state,
                                    oi_social_summary *out_summary);

/* ---- per-term mention counts by time bucket, over the whole vocabulary (docs/SPEC.md §8c) ---
 * out_counts[t * n_buckets + b] = the number of this shard's posts that mention term t and were created in
 * [edges[b], edges[b+1]), for every term t of the BM25 part (n_terms as oi_index_read_bm25 reports it), term-major, host
 * memory.  A post that repeats the term counts once; source: -1 = all posts, else only that source's.  It equals the
 * `total` of oi_index_mention_timeline's state for (t, b), without the sort and the summaries.  A document-sharded
 * index sums the shards' counts (integers: the sum is exact in any order); a shard without a posting returns zeros.
 * OI_ERR_STATE: no BM25 part, no signals or no times loaded.  OI_ERR_INVALID_ARG: NULL edges / out_counts,
 * n_buckets == 0, edges not strictly increasing, source outside -1 .. OI_N_SOURCES - 1.  A refused call changes nothing.
 * OI_ERR_OUT_OF_MEMORY: no room for the counts on the device.  Blocking; reads the posting lists only, so it works
 * before and after oi_index_bm25_finalize. */
oi_status oi_index_mention_counts(oi_index *h, const int64_t *edges, uint32_t n_buckets, int32_t source,
                                  uint32_t *out_counts);

/* ---- tuning / introspection (bench + tests) ------------------------------------------------ */
/* number of kernels this handle has launched since creation (bench "gpu_launches") */
uint64_t oi_index_launch_count(const oi_index *h);
/* named integer knobs: "cosine_variant" (0 = ldg, 1 = bulk-copy pipeline), "cosine_gemm_min_batch"
 * (bf16 batches of at least this many queries take the tcgen05 tensor-core path; 0 = never),
 * "cosine_gemm_cap" (tests: force list compaction), "cosine_gemm_sample_tiles" (probe-pass tiles per CTA; > 0 also forces
 * the probe pass on small shards), "cosine_gemm_pair" (1 = default: an even number of 128-query tiles runs as CTA pairs,
 * tcgen05.mma.cta_group::2 with M = 256; 0 = single CTAs only; same lists bit for bit), "cosine_gemm_pair_ring" (24 | 48);
 * "cosine_multi_query" (2 = default: a call with several queries reads the matrix once per group of 4 queries when a
 * row is at most 1536 bytes, on the bulk-copy pipeline for f32 rows; 1 = same with direct loads; 0 = every query
 * scans the matrix on its own);
 * BM25 schedule: "bm25_warps" (warps per CTA), "bm25_block_docs" (documents per block, power of two >= 1024),
 * "bm25_stage_slots" (TMA-staged 64-posting chunks per warp), "bm25_items_per_warp" (0 = default: 16 per warp and at
 * most 32 blocks per item), "bm25_dense_div" (before
 * finalize: a term in >= n_docs / div documents gets a dense weight column), "bm25_no_cold_bound" (tests);
 * every setting returns the same lists bit for bit.
 * Hybrid call: "hybrid_overlap" (0 = default: the two legs back to back; 1 = BM25 on a second stream next to the
 * GEMM, co-resident "lite" kernels with "overlap_bm25_warps" / "overlap_bm25_slots"; 2 = SM partition with
 * "overlap_gemm_sms"): identical results, measured in profiles/r02_overlap_sweep.md.
 * "cosine_gemm_debug", "cosine_gemm_lite", "comm_debug_skip_gather": timing experiments only. */
oi_status oi_index_set_option(oi_index *h, const char *name, int64_t value);
/* tests: the raw nq x n_docs f32 score matrix of the tensor-core path (bf16 index, small shards) */
oi_status oi_debug_cosine_gemm_scores(oi_index *h, const float *queries, uint32_t nq, float *out_scores);

#ifdef __cplusplus
}
#endif
#endif
