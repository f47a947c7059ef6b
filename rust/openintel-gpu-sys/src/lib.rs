//! `extern "C"` surface of libopenintel_gpu.so — one declaration per entry of include/openintel_gpu.h.
//! UNCOMPILED in the source repository (no Rust toolchain there).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

pub type oi_status = i32;
pub const OI_OK: oi_status = 0;
pub const OI_ERR_INVALID_ARG: oi_status = 1;
pub const OI_ERR_NO_DEVICE: oi_status = 2;
pub const OI_ERR_CUDA: oi_status = 3;
pub const OI_ERR_OUT_OF_MEMORY: oi_status = 4;
pub const OI_ERR_STATE: oi_status = 5;
pub const OI_ERR_COMM: oi_status = 6;
pub const OI_ERR_UNSUPPORTED: oi_status = 7;
pub const OI_NO_DOC: u32 = 0xFFFF_FFFF;
pub const OI_MAX_K: u32 = 1024;
pub const OI_MAX_DIM: u32 = 24576;
pub const OI_UNIQUE_ID_BYTES: usize = 128;
pub const OI_P2P_HANDLE_BYTES: usize = 64;
pub const OI_DTYPE_F32: u32 = 0;
pub const OI_DTYPE_BF16: u32 = 1;
/// post sources in store-schema order: 0 = reddit, 1 = bluesky
pub const OI_N_SOURCES: usize = 2;
/// anchors of one co-mention call: one bit of the per-post mask each (docs/SPEC.md §8d)
pub const OI_MAX_COMENTION_ANCHORS: u32 = 64;

#[repr(C)]
pub struct oi_index {
    _private: [u8; 0],
}

#[repr(C)]
pub struct oi_lexicon {
    _private: [u8; 0],
}

/// SpeculationEngine::social_summary of a batch (src/domain/engine/speculation_engine.rs:70-125)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct oi_social_summary {
    pub total: u64,
    pub bullish: u64,
    pub bearish: u64,
    pub neutral: u64,
    pub net_sentiment: f64,
    pub speculation_index: f64,
    pub bull_bear_ratio: f64,
}

/// the running state of one term's summary after a prefix of the doc order (docs/SPEC.md §8a)
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct oi_mention_state {
    pub total: u64,
    pub bullish: u64,
    pub bearish: u64,
    pub neutral: u64,
    pub speculative: u64,
    pub by_source: [u64; OI_N_SOURCES],
    /// sequential f64 sum of the polarities so far, doc order
    pub sum: f64,
}

/// one (term, author) run of oi_index_mention_authors (docs/SPEC.md §8e); `term` indexes the call's term ids
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct oi_author_run {
    pub term: u32,
    pub author: u32,
    pub posts: u64,
    pub bullish: u64,
    pub bearish: u64,
    pub speculative: u64,
    pub engagement: u64,
    pub first_at: i64,
    pub last_at: i64,
}

#[repr(C)]
pub struct oi_index_desc {
    pub struct_size: u32,
    pub device: i32,
    pub n_docs: u64,
    pub doc_base: u64,
    pub dim: u32,
    pub dtype: u32,
    pub max_k: u32,
    pub max_batch: u32,
}

#[repr(C)]
pub struct oi_bm25_params {
    pub struct_size: u32,
    pub k1: f32,
    pub b: f32,
    pub avgdl: f32,
    pub n_docs_global: u64,
    pub global_df: *const u32,
}

extern "C" {
    pub fn oi_index_create(desc: *const oi_index_desc, out: *mut *mut oi_index) -> oi_status;
    pub fn oi_index_destroy(h: *mut oi_index);
    pub fn oi_last_error(h: *const oi_index) -> *const c_char;
    pub fn oi_version() -> *const c_char;

    pub fn oi_index_load_embeddings(h: *mut oi_index, rows: *const c_void, first_doc: u64, n: u64) -> oi_status;
    pub fn oi_index_synth_embeddings(h: *mut oi_index, seed: u64) -> oi_status;
    pub fn oi_index_read_embeddings(h: *mut oi_index, rows: *mut c_void, first_doc: u64, n: u64) -> oi_status;

    pub fn oi_index_load_bm25(h: *mut oi_index, term_offsets: *const u64, doc_ids: *const u32, tfs: *const u32,
                              doc_len: *const u32, n_terms: u32) -> oi_status;
    pub fn oi_index_synth_bm25(h: *mut oi_index, seed: u64, vocab: u32, zipf_cdf: *const f64) -> oi_status;
    pub fn oi_index_build_bm25_text(h: *mut oi_index, texts: *const u8, offsets: *const u64, n_posts: u64,
                                    out_n_terms: *mut u32, out_vocab_bytes: *mut u64) -> oi_status;
    pub fn oi_index_bm25_union_vocabulary(h: *mut oi_index, terms: *const u8, offsets: *const u64, n_entries: u64,
                                          out_n_terms: *mut u32, out_vocab_bytes: *mut u64) -> oi_status;
    pub fn oi_index_read_vocabulary(h: *mut oi_index, bytes: *mut u8, offsets: *mut u64) -> oi_status;
    pub fn oi_index_bm25_local_stats(h: *mut oi_index, df_out: *mut u32, sum_doc_len: *mut u64, n_postings: *mut u64) -> oi_status;
    pub fn oi_index_bm25_finalize(h: *mut oi_index, params: *const oi_bm25_params) -> oi_status;
    pub fn oi_index_read_bm25(h: *mut oi_index, term_offsets: *mut u64, doc_ids: *mut u32, tfs: *mut u32, doc_len: *mut u32,
                              weights: *mut f32) -> oi_status;

    pub fn oi_comm_unique_id(out: *mut u8) -> oi_status;
    pub fn oi_index_comm_init(h: *mut oi_index, rank: i32, world_size: i32, unique_id: *const u8) -> oi_status;
    pub fn oi_index_p2p_export(h: *mut oi_index, out: *mut u8) -> oi_status;
    pub fn oi_index_p2p_attach(h: *mut oi_index, handles: *const u8) -> oi_status;
    pub fn oi_index_p2p_status(h: *mut oi_index, batches: *mut u64, timed_out: *mut u32) -> oi_status;

    pub fn oi_search_cosine(h: *mut oi_index, queries: *const f32, nq: u32, k: u32, out_ids: *mut u32, out_scores: *mut f32) -> oi_status;
    pub fn oi_search_bm25(h: *mut oi_index, q_terms: *const u32, q_offsets: *const u32, nq: u32, k: u32, out_ids: *mut u32,
                          out_scores: *mut f32) -> oi_status;
    pub fn oi_search_hybrid(h: *mut oi_index, queries: *const f32, q_terms: *const u32, q_offsets: *const u32, nq: u32, k: u32,
                            rrf_k: u32, out_ids: *mut u32, out_rrf: *mut f32, out_rank_cos: *mut u32, out_rank_bm25: *mut u32) -> oi_status;

    pub fn oi_search_cosine_dev(h: *mut oi_index, d_queries: *const f32, nq: u32, k: u32, d_out_ids: *mut u32,
                                d_out_scores: *mut f32, cuda_stream: *mut c_void) -> oi_status;
    pub fn oi_search_bm25_dev(h: *mut oi_index, d_q_terms: *const u32, d_q_offsets: *const u32, nq: u32, k: u32,
                              d_out_ids: *mut u32, d_out_scores: *mut f32, cuda_stream: *mut c_void) -> oi_status;
    pub fn oi_search_hybrid_dev(h: *mut oi_index, d_queries: *const f32, d_q_terms: *const u32, d_q_offsets: *const u32, nq: u32,
                                k: u32, rrf_k: u32, d_out_ids: *mut u32, d_out_rrf: *mut f32, d_out_rank_cos: *mut u32,
                                d_out_rank_bm25: *mut u32, cuda_stream: *mut c_void) -> oi_status;

    pub fn oi_lexicon_analyze(device: i32, texts: *const u8, offsets: *const u64, n_posts: u64, out_polarity: *mut f64,
                              out_speculative: *mut u8, out_bull_hits: *mut u32, out_bear_hits: *mut u32) -> oi_status;

    pub fn oi_lexicon_create(device: i32, reserve_bytes: u64, reserve_posts: u64, out: *mut *mut oi_lexicon) -> oi_status;
    pub fn oi_lexicon_destroy(lx: *mut oi_lexicon);
    pub fn oi_lexicon_run(lx: *mut oi_lexicon, texts: *const u8, offsets: *const u64, n_posts: u64, out_polarity: *mut f64,
                          out_speculative: *mut u8, out_bull_hits: *mut u32, out_bear_hits: *mut u32, bull_bear_threshold: f64,
                          out_summary: *mut oi_social_summary) -> oi_status;
    pub fn oi_lexicon_launch_count(lx: *const oi_lexicon) -> u64;

    pub fn oi_index_load_post_signals(h: *mut oi_index, polarity: *const f64, speculative: *const u8, source: *const u8) -> oi_status;
    pub fn oi_index_mention_summary(h: *mut oi_index, terms: *const u32, n_terms: u32, source: i32, bull_bear_threshold: f64,
                                    carry_in: *const oi_mention_state, out_state: *mut oi_mention_state,
                                    out_summary: *mut oi_social_summary) -> oi_status;
    /// per-post creation times of this shard, seconds since the Unix epoch (docs/SPEC.md §8b)
    pub fn oi_index_load_post_times(h: *mut oi_index, created_at: *const i64) -> oi_status;
    /// per-(term, bucket) summaries, [n_terms][n_buckets] term-major; edges has n_buckets + 1 entries
    pub fn oi_index_mention_timeline(h: *mut oi_index, terms: *const u32, n_terms: u32, edges: *const i64, n_buckets: u32,
                                     source: i32, bull_bear_threshold: f64, carry_in: *const oi_mention_state,
                                     out_state: *mut oi_mention_state, out_summary: *mut oi_social_summary) -> oi_status;
    /// per-(term, bucket) mention counts over every term of the BM25 part, [n_terms][n_buckets] term-major
    /// (docs/SPEC.md §8c); edges has n_buckets + 1 entries
    pub fn oi_index_mention_counts(h: *mut oi_index, edges: *const i64, n_buckets: u32, source: i32,
                                   out_counts: *mut u32) -> oi_status;
    /// co-mention counts of at most OI_MAX_COMENTION_ANCHORS anchors against every term of the BM25 part,
    /// [n_anchors][n_terms] anchor-major, over the posts in window = [since, until) (docs/SPEC.md §8d)
    pub fn oi_index_comention_counts(h: *mut oi_index, anchors: *const u32, n_anchors: u32, window: *const i64, source: i32,
                                     out_counts: *mut u32) -> oi_status;
    /// per pair (anchor_terms[j], terms[j]): the social summary of the posts in the window that mention both, relayed
    /// like oi_index_mention_summary
    pub fn oi_index_comention_summary(h: *mut oi_index, anchor_terms: *const u32, terms: *const u32, n_pairs: u32,
                                      window: *const i64, source: i32, bull_bear_threshold: f64,
                                      carry_in: *const oi_mention_state, out_state: *mut oi_mention_state,
                                      out_summary: *mut oi_social_summary) -> oi_status;
    /// per-post author ids (dense, global) and engagement of this shard (docs/SPEC.md §8e)
    pub fn oi_index_load_post_authors(h: *mut oi_index, author: *const u32, engagement: *const u32) -> oi_status;
    /// the (term, author) runs of the posts in window = [since, until), sorted by (term index, author id); term i's runs
    /// are out_runs[out_term_runs[i] .. out_term_runs[i + 1]); more runs than `capacity`: refused with the count needed
    pub fn oi_index_mention_authors(h: *mut oi_index, terms: *const u32, n_terms: u32, window: *const i64, source: i32,
                                    bull_bear_threshold: f64, capacity: u64, out_term_runs: *mut u64,
                                    out_runs: *mut oi_author_run, out_n_runs: *mut u64) -> oi_status;

    pub fn oi_index_launch_count(h: *const oi_index) -> u64;
    pub fn oi_index_set_option(h: *mut oi_index, name: *const c_char, value: i64) -> oi_status;
    pub fn oi_debug_cosine_gemm_scores(h: *mut oi_index, queries: *const f32, nq: u32, out_scores: *mut f32) -> oi_status;
}
