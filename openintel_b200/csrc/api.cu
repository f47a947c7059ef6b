// api.cu — the extern "C" boundary of libopenintel_gpu.so (include/openintel_gpu.h).
// Owns the index handle, validates arguments, sequences kernels on a stream, and turns every
// failure into a status code + message.  No CPU fallback exists: without a CUDA device the
// library refuses to create an index.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <new>

#include "handle.h"

static thread_local std::string g_create_error;

oi_status oi_index::fail(oi_status code, const char *fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  err = buf;
  return code;
}

#define OI_REQUIRE(cond, ...)                                   \
  do {                                                          \
    if (!(cond)) return h->fail(OI_ERR_INVALID_ARG, __VA_ARGS__); \
  } while (0)

void oi_set_thread_error(const std::string &msg) { g_create_error = msg; }

static oi_status create_fail(oi_status code, const std::string &msg) {
  g_create_error = msg;
  return code;
}

extern "C" const char *oi_version(void) { return "openintel_gpu 0.1 (sm_100a; cosine scan + BM25 + RRF; no CPU fallback)"; }

// The message is copied under the handle's lock into a thread-local string: a failing call on another thread may
// reassign h->err at any time, and the pointer handed out must stay valid until this thread asks again.
extern "C" const char *oi_last_error(const oi_index *h) {
  if (!h) return g_create_error.c_str();
  static thread_local std::string t_msg;
  oi_index *hm = const_cast<oi_index *>(h);
  std::lock_guard<std::mutex> lock(hm->mu);
  t_msg = hm->err;
  return t_msg.c_str();
}

// Device-side ordering of two calls that share the handle's workspaces but were enqueued on different streams
// (ADVICE r1): the stream of this call waits for the event recorded at the end of the previous one.  A capturing
// stream is left alone (the host that captures owns the ordering of its graph).
static bool stream_is_capturing(cudaStream_t st) {
  cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
  if (cudaStreamIsCapturing(st, &cs) != cudaSuccess) { cudaGetLastError(); return false; }
  return cs != cudaStreamCaptureStatusNone;
}
cudaError_t call_begin(oi_index *h, cudaStream_t st) {
  if (!h->has_last || st == h->last_stream || stream_is_capturing(st)) return cudaSuccess;
  return cudaStreamWaitEvent(st, h->ev_last, 0);
}
cudaError_t call_end(oi_index *h, cudaStream_t st) {
  if (stream_is_capturing(st)) return cudaSuccess;
  cudaError_t e = cudaEventRecord(h->ev_last, st);
  if (e == cudaSuccess) { h->has_last = true; h->last_stream = st; }
  return e;
}

extern "C" oi_status oi_index_create(const oi_index_desc *desc, oi_index **out) {
  if (!out) return create_fail(OI_ERR_INVALID_ARG, "out is NULL");
  *out = nullptr;
  if (!desc || desc->struct_size != sizeof(oi_index_desc)) return create_fail(OI_ERR_INVALID_ARG, "bad oi_index_desc (struct_size mismatch)");
  if (desc->dtype != OI_DTYPE_F32 && desc->dtype != OI_DTYPE_BF16) return create_fail(OI_ERR_INVALID_ARG, "dtype must be OI_DTYPE_F32 or OI_DTYPE_BF16");
  const uint32_t esize = desc->dtype == OI_DTYPE_F32 ? 4 : 2;
  if (desc->dim == 0 || (desc->dim * esize) % 16 != 0) return create_fail(OI_ERR_INVALID_ARG, "dim * sizeof(dtype) must be a non-zero multiple of 16 bytes");
  if (desc->max_k == 0 || desc->max_k > OI_MAX_K) return create_fail(OI_ERR_INVALID_ARG, "max_k must be in 1..1024");
  if (desc->max_batch == 0 || desc->max_batch > 65536) return create_fail(OI_ERR_INVALID_ARG, "max_batch must be in 1..65536");
  if (desc->n_docs + desc->doc_base > 0xFFFFFFFEull) return create_fail(OI_ERR_INVALID_ARG, "doc ids must fit in u32 (doc_base + n_docs <= 2^32 - 2)");

  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return create_fail(OI_ERR_NO_DEVICE, std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this library has no CPU fallback)");
  if (desc->device < 0 || desc->device >= n_dev) return create_fail(OI_ERR_INVALID_ARG, "device ordinal out of range");

  oi_index *h = new (std::nothrow) oi_index();
  if (!h) return create_fail(OI_ERR_OUT_OF_MEMORY, "host allocation failed");
  h->desc = *desc;
  auto bail = [&](const char *what, cudaError_t ce) {
    std::string m = std::string(what) + ": " + cudaGetErrorString(ce);
    oi_index_destroy(h);
    return create_fail(ce == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, m);
  };
  if ((e = cudaSetDevice(desc->device)) != cudaSuccess) return bail("cudaSetDevice", e);
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, desc->device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
  if (prop.major != 10) {
    oi_index_destroy(h);
    return create_fail(OI_ERR_UNSUPPORTED, "this build targets sm_100a (B200) only");
  }
  h->num_sms = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaStreamCreateWithFlags(&h->stream2, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
  if ((e = cudaEventCreateWithFlags(&h->ev_last, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  if ((e = cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);

  const size_t emb_bytes = (size_t)desc->n_docs * desc->dim * esize;
  if (emb_bytes && (e = cudaMalloc(&h->d_emb, emb_bytes)) != cudaSuccess) return bail("cudaMalloc(embeddings)", e);

  const size_t B = desc->max_batch, K = desc->max_k;
  h->cws.max_grid = oi_cosine_scan_max_grid(h->num_sms);
  h->cws.k_stride = desc->max_k;
  // one candidate area per query of a batch: the persistent scan launch walks the batch's queries back to back
  // and the epilogue of query i overlaps the scan of query i + 1
  h->cws_slots = B;
  if ((e = cudaMalloc(&h->cws.cand, h->cws_slots * h->cws.max_grid * K * sizeof(u64))) != cudaSuccess) return bail("cudaMalloc(cand)", e);
  if ((e = cudaMalloc(&h->cws.gthr, B * sizeof(u64))) != cudaSuccess) return bail("cudaMalloc(gthr)", e);
  if ((e = cudaMalloc(&h->cws.ticket, B * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc(ticket)", e);
  if ((e = cudaMemset(h->cws.gthr, 0, B * sizeof(u64))) != cudaSuccess) return bail("cudaMemset", e);
  if ((e = cudaMemset(h->cws.ticket, 0, B * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMemset", e);
  if ((e = cudaMalloc(&h->cws.tile_ctr, B * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc(tile_ctr)", e);
  if ((e = cudaMemset(h->cws.tile_ctr, 0, B * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMemset", e);
  if ((e = cudaMalloc(&h->d_queries, B * desc->dim * sizeof(float))) != cudaSuccess) return bail("cudaMalloc(queries)", e);
  if ((e = cudaMalloc(&h->d_keys_cos, B * K * sizeof(u64))) != cudaSuccess) return bail("cudaMalloc(keys)", e);
  if ((e = cudaMalloc(&h->d_keys_bm25, B * K * sizeof(u64))) != cudaSuccess) return bail("cudaMalloc(keys)", e);
  if ((e = cudaMalloc(&h->d_out_u32, 3 * B * K * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc(out)", e);
  if ((e = cudaMalloc(&h->d_out_f32, B * K * sizeof(float))) != cudaSuccess) return bail("cudaMalloc(out)", e);
  for (oi_index::Slot &sl : h->slots) {
    if ((e = cudaHostAlloc(&sl.h_in, OI_PIN_BYTES, cudaHostAllocDefault)) != cudaSuccess) return bail("cudaHostAlloc", e);
    if ((e = cudaHostAlloc(&sl.h_out, OI_PIN_BYTES, cudaHostAllocDefault)) != cudaSuccess) return bail("cudaHostAlloc", e);
    if ((e = cudaMalloc(&sl.d_in, OI_PIN_BYTES)) != cudaSuccess) return bail("cudaMalloc(staging)", e);
    if ((e = cudaMalloc(&sl.d_out, OI_PIN_BYTES)) != cudaSuccess) return bail("cudaMalloc(staging)", e);
    if ((e = cudaEventCreateWithFlags(&sl.done, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
  }
  *out = h;
  return OI_OK;
}

extern "C" void oi_index_destroy(oi_index *h) {
  if (!h) return;
  cudaSetDevice(h->desc.device);
  if (h->stream) cudaStreamSynchronize(h->stream);
  if (h->stream2) cudaStreamSynchronize(h->stream2);
  if (h->has_last) cudaEventSynchronize(h->ev_last);  // a `_dev` call may still be running on a caller's stream
  oi_comm_destroy(h);
  oi_bm25_free(h);
  oi_gemm_free(h);
  oi_mention_free(h);
  cudaFree(h->d_emb);
  cudaFree(h->cws.cand);
  cudaFree(h->cws.gthr);
  cudaFree(h->cws.ticket);
  cudaFree(h->cws.tile_ctr);
  cudaFree(h->d_queries);
  cudaFree(h->d_keys_cos);
  cudaFree(h->d_keys_bm25);
  cudaFree(h->d_out_u32);
  cudaFree(h->d_out_f32);
  cudaFree(h->d_gather);
  for (oi_index::Slot &sl : h->slots) {
    cudaFree(sl.d_in);
    cudaFree(sl.d_out);
    cudaFreeHost(sl.h_in);
    cudaFreeHost(sl.h_out);
    if (sl.done) cudaEventDestroy(sl.done);
  }
  if (h->ev_last) cudaEventDestroy(h->ev_last);
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  if (h->ev_join) cudaEventDestroy(h->ev_join);
  if (h->stream2) cudaStreamDestroy(h->stream2);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

extern "C" uint64_t oi_index_launch_count(const oi_index *h) { return h ? h->launches : 0; }

extern "C" oi_status oi_index_set_option(oi_index *h, const char *name, int64_t value) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OI_REQUIRE(name != nullptr, "option name is NULL");
  if (!strcmp(name, "cosine_variant")) {
    OI_REQUIRE(value == 0 || value == 1, "cosine_variant must be 0 (ldg) or 1 (bulk pipeline)");
    h->cosine_variant = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_multi_query")) {
    OI_REQUIRE(value >= 0 && value <= 2, "cosine_multi_query must be 0 (every query scans the matrix on its own), 1 (direct loads) or 2 (bulk-copy pipeline)");
    h->cosine_multi_query = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_scan_shape")) {  // experiments (process-wide): value = tile_rows * 256 + stages (0 = default)
    // a tile may not hold more rows than half the CTA's candidate buffer, or a cold tile could overflow it
    OI_REQUIRE(value >= 0 && (value >> 8) <= OI_MAX_K && (value & 255) <= 8, "cosine_scan_shape: tile_rows must be <= 1024 and stages <= 8");
    oi_cosine_scan_tuning((int)(value >> 8), (int)(value & 255));
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_pair")) {  // 0: never CTA pairs (every CTA issues its own M = 128 MMAs)
    OI_REQUIRE(value == 0 || value == 1, "cosine_gemm_pair must be 0 or 1");
    h->gemm_pair = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_pair_ring")) {
    OI_REQUIRE(value == 24 || value == 48, "cosine_gemm_pair_ring must be 24 or 48");
    h->gemm_pair_ring = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_lite")) {  // experiments: the stand-alone cosine call runs the 96 KB-ring kernel too
    h->gemm_force_lite = value != 0;
    return OI_OK;
  }
  if (!strcmp(name, "hybrid_overlap")) {
    OI_REQUIRE(value >= 0 && value <= 2, "hybrid_overlap must be 0 (legs back to back), 1 (co-resident lite kernels) or 2 (SM partition)");
    h->hybrid_overlap = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "overlap_bm25_warps")) {
    OI_REQUIRE(value >= 1 && value <= 16, "overlap_bm25_warps must be in 1..16");
    h->overlap_bm25_warps = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "overlap_bm25_slots")) {
    OI_REQUIRE(value >= 0 && value <= 8, "overlap_bm25_slots must be in 0..8");
    h->overlap_bm25_slots = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "overlap_gemm_sms")) {
    OI_REQUIRE(value >= 2 && value < h->num_sms, "overlap_gemm_sms must be in 2..num_sms-1");
    h->overlap_gemm_sms = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_min_batch")) {
    OI_REQUIRE(value >= 0 && value <= 65536, "cosine_gemm_min_batch must be in 0..65536 (0 = tensor-core path off)");
    h->gemm_min_batch = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_force_2d")) {
    h->gemm_force_2d = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_debug")) {  // timing experiments: results are garbage while it is set
    OI_REQUIRE(value >= 0 && value <= 15, "cosine_gemm_debug is a 4-bit mask");
    h->gemm_debug = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_cap")) {
    OI_REQUIRE(value == 0 || value == 128 || value == 256 || value == 512, "cosine_gemm_cap must be 0, 128, 256 or 512");
    h->gemm_cap = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "cosine_gemm_sample_tiles")) {
    OI_REQUIRE(value >= 0 && value <= 56, "cosine_gemm_sample_tiles must be in 0..56");
    h->gemm_sample_tiles = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "no_pinned_staging")) {
    h->no_pinned_staging = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "comm_exchange")) {  // 0 = ncclAllGather, 1 = peer-to-peer push (needs oi_index_p2p_attach)
    OI_REQUIRE(value == 0 || value == 1, "comm_exchange must be 0 (NCCL all-gather) or 1 (peer-to-peer push)");
    h->comm_exchange = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "comm_debug_skip_gather")) {
    h->comm_skip = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "bm25_variant")) {
    h->bm25_variant = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "bm25_warps")) {
    OI_REQUIRE(value >= 0 && value <= 24, "bm25_warps must be in 0..24 (0 = default)");
    h->bm25_warps = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "bm25_block_docs")) {
    OI_REQUIRE(value == 0 || (value >= 1024 && value <= 32768 && (value & (value - 1)) == 0), "bm25_block_docs must be 0 or a power of two in 1024..32768");
    h->bm25_block_docs = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "bm25_dense_div")) {
    OI_REQUIRE(value >= 0 && value <= 1024, "bm25_dense_div must be in 0..1024 (0 = default)");
    h->bm25_dense_div = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "bm25_items_per_warp")) {
    OI_REQUIRE(value >= 0 && value <= 256, "bm25_items_per_warp must be in 0..256 (0 = default)");
    h->bm25_items_per_warp = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "bm25_no_cold_bound")) {
    h->bm25_no_cold_bound = (int)value;
    return OI_OK;
  }
  if (!strcmp(name, "bm25_stage_slots")) {
    OI_REQUIRE(value >= -1 && value <= 16, "bm25_stage_slots must be in -1..16 (-1 = default)");
    h->bm25_stage_slots = (int)value;
    return OI_OK;
  }
  return h->fail(OI_ERR_INVALID_ARG, "unknown option '%s'", name);
}

// ---- embeddings -------------------------------------------------------------------------------
extern "C" oi_status oi_index_load_embeddings(oi_index *h, const void *rows, uint64_t first_doc, uint64_t n) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OI_REQUIRE(rows != nullptr || n == 0, "rows is NULL");
  OI_REQUIRE(first_doc + n <= h->desc.n_docs, "rows [%llu, %llu) outside the shard (n_docs = %llu)",
             (unsigned long long)first_doc, (unsigned long long)(first_doc + n), (unsigned long long)h->desc.n_docs);
  // coverage, not a row count: chunks extend the loaded prefix [0, emb_rows_loaded) or rewrite rows inside it, so
  // "all rows loaded" can never be claimed while part of the matrix is uninitialised HBM
  if (first_doc > h->emb_rows_loaded)
    return h->fail(OI_ERR_STATE, "rows [%llu, ...) would leave a gap after the %llu rows loaded so far: load chunks in order",
                   (unsigned long long)first_doc, (unsigned long long)h->emb_rows_loaded);
  OI_CK(cudaSetDevice(h->desc.device));
  const size_t row_bytes = (size_t)h->desc.dim * h->esize();
  OI_CK(call_begin(h, h->stream));
  if (n) OI_CK(cudaMemcpyAsync((char *)h->d_emb + first_doc * row_bytes, rows, n * row_bytes, cudaMemcpyHostToDevice, h->stream));
  OI_CK(cudaStreamSynchronize(h->stream));
  if (first_doc + n > h->emb_rows_loaded) h->emb_rows_loaded = first_doc + n;
  return OI_OK;
}

extern "C" oi_status oi_index_synth_embeddings(oi_index *h, uint64_t seed) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OI_CK(cudaSetDevice(h->desc.device));
  OI_CK(call_begin(h, h->stream));
  OI_CK(oi_launch_synth_embeddings(h->d_emb, h->desc.dtype, h->desc.n_docs, h->desc.dim, seed, 0, h->desc.doc_base, h->stream, &h->launches));
  OI_CK(cudaStreamSynchronize(h->stream));
  h->emb_rows_loaded = h->desc.n_docs;
  return OI_OK;
}

extern "C" oi_status oi_index_read_embeddings(oi_index *h, void *rows, uint64_t first_doc, uint64_t n) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OI_REQUIRE(rows != nullptr || n == 0, "rows is NULL");
  OI_REQUIRE(first_doc + n <= h->desc.n_docs, "rows outside the shard");
  OI_CK(cudaSetDevice(h->desc.device));
  const size_t row_bytes = (size_t)h->desc.dim * h->esize();
  OI_CK(call_begin(h, h->stream));
  if (n) OI_CK(cudaMemcpyAsync(rows, (const char *)h->d_emb + first_doc * row_bytes, n * row_bytes, cudaMemcpyDeviceToHost, h->stream));
  OI_CK(cudaStreamSynchronize(h->stream));
  return OI_OK;
}

// ---- search -----------------------------------------------------------------------------------
static oi_status check_search_args(oi_index *h, uint32_t nq, uint32_t k) {
  OI_REQUIRE(k >= 1 && k <= h->desc.max_k, "k = %u outside 1..max_k (%u)", k, h->desc.max_k);
  OI_REQUIRE(nq <= h->desc.max_batch, "nq = %u exceeds max_batch (%u)", nq, h->desc.max_batch);
  return OI_OK;
}

static bool use_gemm(const oi_index *h, uint32_t nq, uint32_t k) {
  return h->gemm_min_batch > 0 && nq >= (uint32_t)h->gemm_min_batch && oi_gemm_eligible(h, nq, k);
}

// local scan -> (multi-GPU: all-gather + merge) -> global cosine key lists in d_keys_cos
// `local_only` (multi-GPU hybrid): leave the shard-local lists there and skip the exchange
// gemm_lite / gemm_ctas: the hybrid call's overlap modes (see hybrid_enqueue)
static oi_status cosine_keys(oi_index *h, const float *d_queries, uint32_t nq, uint32_t k, cudaStream_t st, u64 *local_only = nullptr,
                             bool gemm_lite = false, uint32_t gemm_ctas = 0) {
  if (h->emb_rows_loaded < h->desc.n_docs) return h->fail(OI_ERR_STATE, "embeddings not loaded (%llu of %llu rows)", (unsigned long long)h->emb_rows_loaded, (unsigned long long)h->desc.n_docs);
  if (nq == 0) return OI_OK;
  u64 *local = local_only ? local_only : (h->world > 1 ? h->d_keys_local : h->d_keys_cos);
  if (use_gemm(h, nq, k)) {
    // batched bf16 queries: one pass of the matrix through the tensor cores serves the whole batch
    oi_status s = oi_gemm_local_keys(h, d_queries, nq, k, local, nullptr, st, gemm_lite || h->gemm_force_lite, gemm_ctas);
    if (s) return s;
  } else {
    OI_CK(oi_launch_cosine_scan(h->d_emb, h->desc.dtype, h->desc.n_docs, h->desc.dim, (uint32_t)h->desc.doc_base, d_queries, nq, k,
                                h->cws, local, h->cosine_variant, h->num_sms, st, &h->launches, h->cosine_multi_query));
  }
  if (h->world > 1 && !local_only) return oi_comm_gather_merge(h, local, nq, k, h->d_keys_cos, st);
  return OI_OK;
}

extern "C" oi_status oi_search_cosine_dev(oi_index *h, const float *d_queries, uint32_t nq, uint32_t k,
                                          uint32_t *d_out_ids, float *d_out_scores, void *cuda_stream) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  oi_status s = check_search_args(h, nq, k);
  if (s) return s;
  OI_REQUIRE(nq == 0 || (d_queries && d_out_ids && d_out_scores), "NULL device pointer");
  if (nq == 0) return OI_OK;
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  OI_CK(call_begin(h, st));
  if ((s = cosine_keys(h, d_queries, nq, k, st))) return s;
  OI_CK(oi_launch_unpack_keys(h->d_keys_cos, nq * k, d_out_ids, d_out_scores, st, &h->launches));
  OI_CK(call_end(h, st));
  return OI_OK;
}

extern "C" oi_status oi_search_cosine(oi_index *h, const float *queries, uint32_t nq, uint32_t k,
                                      uint32_t *out_ids, float *out_scores) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::unique_lock<std::mutex> lock(h->mu);
  oi_status s = check_search_args(h, nq, k);
  if (s) return s;
  OI_REQUIRE(nq == 0 || (queries && out_ids && out_scores), "NULL host pointer");
  if (nq == 0) return OI_OK;
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));
  const size_t qbytes = (size_t)nq * h->desc.dim * sizeof(float), n = (size_t)nq * k;
  if (!h->no_pinned_staging && qbytes <= OI_PIN_BYTES && n * 8 <= OI_PIN_BYTES) {  // small call: one pinned copy each way
    SlotLease lease(h, lock);
    oi_index::Slot *sl = lease.sl;
    memcpy(sl->h_in, queries, qbytes);
    OI_CK(cudaMemcpyAsync(sl->d_in, sl->h_in, qbytes, cudaMemcpyHostToDevice, st));
    if ((s = cosine_keys(h, reinterpret_cast<const float *>(sl->d_in), nq, k, st))) return s;
    uint32_t *d_ids = reinterpret_cast<uint32_t *>(sl->d_out);
    float *d_sc = reinterpret_cast<float *>(sl->d_out + n * 4);
    OI_CK(oi_launch_unpack_keys(h->d_keys_cos, nq * k, d_ids, d_sc, st, &h->launches));
    OI_CK(cudaMemcpyAsync(sl->h_out, sl->d_out, n * 8, cudaMemcpyDeviceToHost, st));
    if ((s = lease.finish(st))) return s;
    memcpy(out_ids, sl->h_out, n * 4);
    memcpy(out_scores, sl->h_out + n * 4, n * 4);
    return OI_OK;
  }
  OI_CK(cudaMemcpyAsync(h->d_queries, queries, qbytes, cudaMemcpyHostToDevice, st));
  if ((s = cosine_keys(h, h->d_queries, nq, k, st))) return s;
  OI_CK(oi_launch_unpack_keys(h->d_keys_cos, nq * k, h->d_out_u32, h->d_out_f32, st, &h->launches));
  OI_CK(cudaMemcpyAsync(out_ids, h->d_out_u32, (size_t)nq * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_scores, h->d_out_f32, (size_t)nq * k * sizeof(float), cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

extern "C" oi_status oi_debug_cosine_gemm_scores(oi_index *h, const float *queries, uint32_t nq, float *out_scores) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OI_REQUIRE(queries && out_scores && nq >= 1 && nq <= h->desc.max_batch, "bad arguments");
  if (!oi_gemm_eligible(h, nq, 1)) return h->fail(OI_ERR_UNSUPPORTED, "tensor-core path needs a bf16 index with dim %% 64 == 0 and dim <= 768");
  if (h->emb_rows_loaded < h->desc.n_docs) return h->fail(OI_ERR_STATE, "embeddings not loaded");
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));
  float *d_dump = nullptr;
  const size_t n = (size_t)nq * h->desc.n_docs;
  OI_CK(cudaMalloc(&d_dump, n * sizeof(float)));
  cudaError_t e = cudaMemcpyAsync(h->d_queries, queries, (size_t)nq * h->desc.dim * sizeof(float), cudaMemcpyHostToDevice, st);
  oi_status s = OI_OK;
  if (e == cudaSuccess) s = oi_gemm_local_keys(h, h->d_queries, nq, 1, h->d_keys_cos, d_dump, st);
  if (e == cudaSuccess && s == OI_OK) e = cudaMemcpyAsync(out_scores, d_dump, n * sizeof(float), cudaMemcpyDeviceToHost, st);
  if (e == cudaSuccess && s == OI_OK) e = cudaStreamSynchronize(st);
  cudaFree(d_dump);
  if (s) return s;
  OI_CK(e);
  return OI_OK;
}

// local BM25 lists -> (multi-GPU: all-gather + merge) -> global BM25 key lists in d_keys_bm25
static oi_status bm25_keys(oi_index *h, const uint32_t *d_terms, const uint32_t *d_offs, uint32_t nq, uint32_t k, cudaStream_t st,
                           u64 *local_only = nullptr, int overlap = 0) {
  if (nq == 0) return OI_OK;
  u64 *local = local_only ? local_only : (h->world > 1 ? h->d_keys_local : h->d_keys_bm25);
  oi_status s = oi_bm25_local_keys(h, d_terms, d_offs, nq, k, local, st, overlap);
  if (s) return s;
  if (h->world > 1 && !local_only) return oi_comm_gather_merge(h, local, nq, k, h->d_keys_bm25, st);
  return OI_OK;
}

// validates the host-side query term arrays.  A query may carry any number of raw term ids: the device de-duplicates
// them in first-seen order and scores at most the first 64 distinct known terms (SPEC §3) -- the same rule the `_dev`
// entry points apply, so both paths return the same lists for the same arrays.  Only the size of the whole call is
// bounded (by the staging array).
static oi_status check_terms(oi_index *h, const uint32_t *q_terms, const uint32_t *q_offsets, uint32_t nq) {
  if (!oi_bm25_stage_terms(h)) return h->fail(OI_ERR_STATE, "no BM25 index loaded");
  OI_REQUIRE(q_offsets != nullptr, "q_offsets is NULL");
  OI_REQUIRE(q_offsets[0] == 0, "q_offsets[0] must be 0");
  for (uint32_t j = 0; j < nq; ++j) OI_REQUIRE(q_offsets[j + 1] >= q_offsets[j], "q_offsets not monotone at query %u", j);
  OI_REQUIRE(q_offsets[nq] == 0 || q_terms != nullptr, "q_terms is NULL");
  OI_REQUIRE(q_offsets[nq] <= oi_bm25_stage_capacity(h), "the call carries %u term ids; at most %llu fit (64 x max_batch)", q_offsets[nq],
             (unsigned long long)oi_bm25_stage_capacity(h));
  return OI_OK;
}

// ... and stages them on the device (the large-call path; small calls pack them into the pinned block)
static oi_status stage_terms(oi_index *h, const uint32_t *q_terms, const uint32_t *q_offsets, uint32_t nq, cudaStream_t st) {
  const uint32_t total = q_offsets[nq];
  if (total) OI_CK(cudaMemcpyAsync(oi_bm25_stage_terms(h), q_terms, (size_t)total * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  OI_CK(cudaMemcpyAsync(oi_bm25_stage_offs(h), q_offsets, ((size_t)nq + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  return OI_OK;
}

// layout of the pinned input block: [queries f32 nq x dim (may be absent)] [offsets u32 nq + 1] [terms u32 total],
// every section 16-byte aligned.  Returns the total size, 0 if it does not fit.
static size_t pin_in_layout(size_t qbytes, uint32_t nq, uint32_t total_terms, size_t *off_offs, size_t *off_terms) {
  const size_t a = (qbytes + 15) & ~(size_t)15;
  const size_t b = a + ((((size_t)nq + 1) * 4 + 15) & ~(size_t)15);
  const size_t c = b + (((size_t)total_terms * 4 + 15) & ~(size_t)15);
  *off_offs = a;
  *off_terms = b;
  return c <= OI_PIN_BYTES ? (c ? c : 16) : 0;
}

extern "C" oi_status oi_search_bm25_dev(oi_index *h, const uint32_t *d_q_terms, const uint32_t *d_q_offsets, uint32_t nq,
                                        uint32_t k, uint32_t *d_out_ids, float *d_out_scores, void *cuda_stream) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  oi_status s = check_search_args(h, nq, k);
  if (s) return s;
  OI_REQUIRE(nq == 0 || (d_q_terms && d_q_offsets && d_out_ids && d_out_scores), "NULL device pointer");
  if (nq == 0) return OI_OK;
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  OI_CK(call_begin(h, st));
  if ((s = bm25_keys(h, d_q_terms, d_q_offsets, nq, k, st))) return s;
  OI_CK(oi_launch_unpack_keys(h->d_keys_bm25, nq * k, d_out_ids, d_out_scores, st, &h->launches));
  OI_CK(call_end(h, st));
  return OI_OK;
}

extern "C" oi_status oi_search_bm25(oi_index *h, const uint32_t *q_terms, const uint32_t *q_offsets, uint32_t nq,
                                    uint32_t k, uint32_t *out_ids, float *out_scores) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::unique_lock<std::mutex> lock(h->mu);
  oi_status s = check_search_args(h, nq, k);
  if (s) return s;
  if (nq == 0) return OI_OK;
  OI_REQUIRE(out_ids && out_scores, "NULL host pointer");
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  if ((s = check_terms(h, q_terms, q_offsets, nq))) return s;
  OI_CK(call_begin(h, st));
  const size_t n = (size_t)nq * k;
  size_t o_offs, o_terms;
  const size_t in_bytes = pin_in_layout(0, nq, q_offsets[nq], &o_offs, &o_terms);
  if (!h->no_pinned_staging && in_bytes && n * 8 <= OI_PIN_BYTES) {  // small call: one pinned copy each way
    SlotLease lease(h, lock);
    oi_index::Slot *sl = lease.sl;
    memcpy(sl->h_in + o_offs, q_offsets, ((size_t)nq + 1) * 4);
    if (q_offsets[nq]) memcpy(sl->h_in + o_terms, q_terms, (size_t)q_offsets[nq] * 4);
    OI_CK(cudaMemcpyAsync(sl->d_in, sl->h_in, in_bytes, cudaMemcpyHostToDevice, st));
    if ((s = bm25_keys(h, reinterpret_cast<const uint32_t *>(sl->d_in + o_terms), reinterpret_cast<const uint32_t *>(sl->d_in + o_offs), nq, k, st))) return s;
    OI_CK(oi_launch_unpack_keys(h->d_keys_bm25, nq * k, reinterpret_cast<uint32_t *>(sl->d_out), reinterpret_cast<float *>(sl->d_out + n * 4), st, &h->launches));
    OI_CK(cudaMemcpyAsync(sl->h_out, sl->d_out, n * 8, cudaMemcpyDeviceToHost, st));
    if ((s = lease.finish(st))) return s;
    memcpy(out_ids, sl->h_out, n * 4);
    memcpy(out_scores, sl->h_out + n * 4, n * 4);
    return OI_OK;
  }
  if ((s = stage_terms(h, q_terms, q_offsets, nq, st))) return s;
  if ((s = bm25_keys(h, oi_bm25_stage_terms(h), oi_bm25_stage_offs(h), nq, k, st))) return s;
  OI_CK(oi_launch_unpack_keys(h->d_keys_bm25, nq * k, h->d_out_u32, h->d_out_f32, st, &h->launches));
  OI_CK(cudaMemcpyAsync(out_ids, h->d_out_u32, (size_t)nq * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_scores, h->d_out_f32, (size_t)nq * k * sizeof(float), cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

// cosine lists + BM25 lists (each global) -> RRF.
//
// The two legs are independent until the fusion.  hybrid_overlap = 0 enqueues them back to back on the caller's stream.
// With the tensor-core cosine path the legs are complementary (GEMM: tensor pipe + HBM, 6 warps; BM25: issue slots +
// L2, no tensor work), so the other modes fork the BM25 leg onto the handle's second stream and join before the
// exchange / fusion:
//   1  co-residency: the GEMM runs its "lite" kernel (96 KB ring, < 128 registers) and the BM25 kernel a CTA of
//      overlap_bm25_warps warps (128 registers), so that ONE CTA OF EACH fits every SM (shared memory 116 + 106 KB,
//      registers 24.5 k + 41 k of 64 k).  The GEMM is launched first: its CTAs take their SMs, the BM25 CTAs fill in.
//   2  SM partition: the stand-alone kernels, the GEMM confined to overlap_gemm_sms SMs, BM25 to the rest.
static oi_status hybrid_enqueue(oi_index *h, const float *d_queries, const uint32_t *d_terms, const uint32_t *d_offs,
                                uint32_t nq, uint32_t k, uint32_t rrf_k, uint32_t *d_ids, float *d_rrf, uint32_t *d_rc,
                                uint32_t *d_rb, cudaStream_t st) {
  oi_status s;
  int mode = h->hybrid_overlap;
  if (mode && (!use_gemm(h, nq, k) || stream_is_capturing(st))) mode = 0;  // the scan path owns every SM: nothing to overlap with
  if (mode == 1 && !oi_gemm_lite_ok(h)) mode = 0;
  const bool sharded = h->world > 1;
  u64 *loc_cos = sharded ? h->d_keys_local : nullptr, *loc_bm = sharded ? h->d_keys_local + (size_t)nq * k : nullptr;
  if (mode) {
    cudaStream_t s2 = h->stream2;
    OI_CK(cudaEventRecord(h->ev_fork, st));
    OI_CK(cudaStreamWaitEvent(s2, h->ev_fork, 0));
    const uint32_t gemm_ctas = mode == 2 ? (uint32_t)h->overlap_gemm_sms : 0u;
    if ((s = cosine_keys(h, d_queries, nq, k, st, loc_cos, mode == 1, gemm_ctas))) return s;
    if ((s = bm25_keys(h, d_terms, d_offs, nq, k, s2, loc_bm, mode))) return s;
    OI_CK(cudaEventRecord(h->ev_join, s2));
    OI_CK(cudaStreamWaitEvent(st, h->ev_join, 0));
    if (sharded) {
      if ((s = oi_comm_gather_merge2(h, h->d_keys_local, nq, k, h->d_keys_cos, h->d_keys_bm25, st))) return s;
    }
  } else if (sharded) {
    // sharded: both local lists first, then ONE exchange for the two modalities (SPEC §5: RRF on the global ranks)
    if ((s = cosine_keys(h, d_queries, nq, k, st, loc_cos))) return s;
    if ((s = bm25_keys(h, d_terms, d_offs, nq, k, st, loc_bm))) return s;
    if ((s = oi_comm_gather_merge2(h, h->d_keys_local, nq, k, h->d_keys_cos, h->d_keys_bm25, st))) return s;
  } else {
    if ((s = cosine_keys(h, d_queries, nq, k, st))) return s;
    if ((s = bm25_keys(h, d_terms, d_offs, nq, k, st))) return s;
  }
  OI_CK(oi_launch_rrf(h->d_keys_cos, h->d_keys_bm25, nq, k, rrf_k, d_ids, d_rrf, d_rc, d_rb, st, &h->launches));
  return OI_OK;
}

extern "C" oi_status oi_search_hybrid_dev(oi_index *h, const float *d_queries, const uint32_t *d_q_terms,
                                          const uint32_t *d_q_offsets, uint32_t nq, uint32_t k, uint32_t rrf_k,
                                          uint32_t *d_out_ids, float *d_out_rrf, uint32_t *d_out_rank_cos,
                                          uint32_t *d_out_rank_bm25, void *cuda_stream) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  oi_status s = check_search_args(h, nq, k);
  if (s) return s;
  OI_REQUIRE(rrf_k >= 1 && rrf_k <= 1000000, "rrf_k = %u outside 1..1e6", rrf_k);
  OI_REQUIRE(nq == 0 || (d_queries && d_q_terms && d_q_offsets && d_out_ids && d_out_rrf && d_out_rank_cos && d_out_rank_bm25), "NULL device pointer");
  if (nq == 0) return OI_OK;
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = (cudaStream_t)cuda_stream;
  OI_CK(call_begin(h, st));
  if ((s = hybrid_enqueue(h, d_queries, d_q_terms, d_q_offsets, nq, k, rrf_k, d_out_ids, d_out_rrf, d_out_rank_cos, d_out_rank_bm25, st))) return s;
  OI_CK(call_end(h, st));
  return OI_OK;
}

extern "C" oi_status oi_search_hybrid(oi_index *h, const float *queries, const uint32_t *q_terms, const uint32_t *q_offsets,
                                      uint32_t nq, uint32_t k, uint32_t rrf_k, uint32_t *out_ids, float *out_rrf,
                                      uint32_t *out_rank_cos, uint32_t *out_rank_bm25) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::unique_lock<std::mutex> lock(h->mu);
  oi_status s = check_search_args(h, nq, k);
  if (s) return s;
  OI_REQUIRE(rrf_k >= 1 && rrf_k <= 1000000, "rrf_k = %u outside 1..1e6", rrf_k);
  if (nq == 0) return OI_OK;
  OI_REQUIRE(queries && out_ids && out_rrf && out_rank_cos && out_rank_bm25, "NULL host pointer");
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  const size_t n = (size_t)nq * k, BK = (size_t)h->desc.max_batch * h->desc.max_k;
  const size_t qbytes = (size_t)nq * h->desc.dim * sizeof(float);
  if ((s = check_terms(h, q_terms, q_offsets, nq))) return s;
  OI_CK(call_begin(h, st));
  size_t o_offs, o_terms;
  const size_t in_bytes = pin_in_layout(qbytes, nq, q_offsets[nq], &o_offs, &o_terms);
  if (!h->no_pinned_staging && in_bytes && n * 16 <= OI_PIN_BYTES) {  // small call: one pinned copy each way
    SlotLease lease(h, lock);
    oi_index::Slot *sl = lease.sl;
    memcpy(sl->h_in, queries, qbytes);
    memcpy(sl->h_in + o_offs, q_offsets, ((size_t)nq + 1) * 4);
    if (q_offsets[nq]) memcpy(sl->h_in + o_terms, q_terms, (size_t)q_offsets[nq] * 4);
    OI_CK(cudaMemcpyAsync(sl->d_in, sl->h_in, in_bytes, cudaMemcpyHostToDevice, st));
    uint32_t *d_ids = reinterpret_cast<uint32_t *>(sl->d_out), *d_rc = d_ids + 2 * n, *d_rb = d_ids + 3 * n;
    float *d_rrf = reinterpret_cast<float *>(d_ids + n);
    if ((s = hybrid_enqueue(h, reinterpret_cast<const float *>(sl->d_in), reinterpret_cast<const uint32_t *>(sl->d_in + o_terms),
                            reinterpret_cast<const uint32_t *>(sl->d_in + o_offs), nq, k, rrf_k, d_ids, d_rrf, d_rc, d_rb, st)))
      return s;
    OI_CK(cudaMemcpyAsync(sl->h_out, sl->d_out, n * 16, cudaMemcpyDeviceToHost, st));
    if ((s = lease.finish(st))) return s;
    memcpy(out_ids, sl->h_out, n * 4);
    memcpy(out_rrf, sl->h_out + n * 4, n * 4);
    memcpy(out_rank_cos, sl->h_out + n * 8, n * 4);
    memcpy(out_rank_bm25, sl->h_out + n * 12, n * 4);
    return OI_OK;
  }
  OI_CK(cudaMemcpyAsync(h->d_queries, queries, qbytes, cudaMemcpyHostToDevice, st));
  if ((s = stage_terms(h, q_terms, q_offsets, nq, st))) return s;
  uint32_t *d_ids = h->d_out_u32, *d_rc = h->d_out_u32 + BK, *d_rb = h->d_out_u32 + 2 * BK;
  if ((s = hybrid_enqueue(h, h->d_queries, oi_bm25_stage_terms(h), oi_bm25_stage_offs(h), nq, k, rrf_k, d_ids, h->d_out_f32, d_rc, d_rb, st))) return s;
  OI_CK(cudaMemcpyAsync(out_ids, d_ids, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_rrf, h->d_out_f32, n * sizeof(float), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_rank_cos, d_rc, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_rank_bm25, d_rb, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}
