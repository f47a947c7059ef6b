// mention.cu — per-term social summaries over the BM25 posting lists (docs/SPEC.md §8a).
//
// A post mentions term t iff one of its tokens equals t: the posts that mention t are t's posting list, doc ids
// ascending.  The handle keeps one lexicon signal per post next to the BM25 part (polarity f64, speculative | source << 1
// in a byte), and one launch runs the shared summary body (oi_summary.cuh) once per requested term, one CTA each, over
// the signals gathered through the term's doc ids.  Every term's chain runs next to the others, so a batch costs about
// its longest list's chain (one dependent DADD per mentioning post with a non-zero polarity); the gather hides behind the
// chain in the tile ring.  The running state in and out lets the shards of a document-sharded index continue one
// another's sequential sum in rank order (a relay), which keeps the mean bit-identical to the unsharded one.
#include <cstring>
#include <vector>

#include "handle.h"
#include "oi_summary.cuh"

namespace {

__global__ void __launch_bounds__(128) mention_summary_kernel(const double *polarity, const uint8_t *flags, const u64 *term_off,
                                                              const uint32_t *doc_ids, const uint32_t *terms, uint32_t n_terms,
                                                              int source, double thr, const oi_mention_state *carry,
                                                              oi_mention_state *out_state, oi_social_summary *out) {
  for (uint32_t i = blockIdx.x; i < n_terms; i += gridDim.x) {
    const u64 lo = term_off[terms[i]], hi = term_off[terms[i] + 1];
    oi_social_summary_cta<true>(polarity, flags, doc_ids, lo, hi - lo, source, thr, carry ? carry + i : nullptr, out_state + i,
                                out + i);
  }
}

size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

}  // namespace

#define MN_CK(call)                                                                              \
  do {                                                                                           \
    cudaError_t e_ = (call);                                                                     \
    if (e_ != cudaSuccess)                                                                       \
      return h->fail(e_ == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA,       \
                     "%s failed: %s", #call, cudaGetErrorString(e_));                            \
  } while (0)

void oi_mention_free(oi_index *h) {
  cudaFree(h->d_sig_pol);
  cudaFree(h->d_sig_flags);
  cudaFree(h->d_mention_io);
  h->d_sig_pol = nullptr;
  h->d_sig_flags = nullptr;
  h->d_mention_io = nullptr;
  h->mention_io_bytes = 0;
  h->has_signals = false;
}

extern "C" oi_status oi_index_load_post_signals(oi_index *h, const double *polarity, const uint8_t *speculative,
                                                const uint8_t *source) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  if (!polarity || !speculative || !source) return h->fail(OI_ERR_INVALID_ARG, "NULL polarity / speculative / source");
  const u64 n = h->desc.n_docs;
  // checked and packed on the host before anything on the device changes: a refused call keeps the previous signals
  std::vector<double> pol(n ? n : 1);
  std::vector<uint8_t> fl(n ? n : 1);
  for (u64 i = 0; i < n; ++i) {
    const double p = polarity[i];
    if (!(p >= -1.0 && p <= 1.0))
      return h->fail(OI_ERR_INVALID_ARG, "post %llu: polarity %g is not a number in [-1, 1]", (unsigned long long)i, p);
    if (speculative[i] > 1)
      return h->fail(OI_ERR_INVALID_ARG, "post %llu: speculative = %u, not 0 / 1", (unsigned long long)i, (unsigned)speculative[i]);
    if (source[i] >= OI_N_SOURCES)
      return h->fail(OI_ERR_INVALID_ARG, "post %llu: source code %u, at most %d", (unsigned long long)i, (unsigned)source[i],
                     OI_N_SOURCES - 1);
    pol[i] = p == 0.0 ? 0.0 : p;  // -0.0 -> +0.0: the summary leaves zero polarities out of its add chain
    fl[i] = (uint8_t)(speculative[i] | source[i] << 1);
  }
  MN_CK(cudaSetDevice(h->desc.device));
  if (!h->d_sig_pol) {
    cudaError_t e = cudaMalloc(&h->d_sig_pol, pol.size() * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_sig_flags, fl.size());
    if (e != cudaSuccess) {
      cudaFree(h->d_sig_pol);
      h->d_sig_pol = nullptr;
      h->d_sig_flags = nullptr;
      return h->fail(e == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, "allocating the post signals failed: %s",
                     cudaGetErrorString(e));
    }
  }
  MN_CK(call_begin(h, h->stream));
  h->has_signals = false;  // until the copies have landed
  if (n) {
    MN_CK(cudaMemcpyAsync(h->d_sig_pol, pol.data(), n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    MN_CK(cudaMemcpyAsync(h->d_sig_flags, fl.data(), n, cudaMemcpyHostToDevice, h->stream));
  }
  MN_CK(call_end(h, h->stream));
  MN_CK(cudaStreamSynchronize(h->stream));
  h->has_signals = true;
  return OI_OK;
}

extern "C" oi_status oi_index_mention_summary(oi_index *h, const uint32_t *terms, uint32_t n_terms, int32_t source,
                                              double bull_bear_threshold, const oi_mention_state *carry_in,
                                              oi_mention_state *out_state, oi_social_summary *out_summary) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::unique_lock<std::mutex> lock(h->mu);
  const u64 *term_off = oi_bm25_term_offsets(h);
  if (!term_off) return h->fail(OI_ERR_STATE, "no BM25 part: the posting lists are the mentions");
  if (!h->has_signals) return h->fail(OI_ERR_STATE, "no post signals loaded (oi_index_load_post_signals)");
  if (n_terms == 0) return OI_OK;
  if (!terms || !out_summary) return h->fail(OI_ERR_INVALID_ARG, "NULL terms / out_summary");
  if (source < -1 || source >= OI_N_SOURCES)
    return h->fail(OI_ERR_INVALID_ARG, "source = %d: -1 (all posts) or a source code below %d", source, OI_N_SOURCES);
  const uint32_t V = oi_bm25_n_terms(h);
  for (uint32_t i = 0; i < n_terms; ++i)
    if (terms[i] >= V) return h->fail(OI_ERR_INVALID_ARG, "terms[%u] = %u: the BM25 part has %u terms", i, terms[i], V);
  MN_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  MN_CK(call_begin(h, st));
  // in: terms u32 [n] | carries [n] (when given); out: states [n] | summaries [n]
  const size_t n = n_terms, o_carry = align16(n * sizeof(uint32_t));
  const size_t in_bytes = o_carry + (carry_in ? n * sizeof(oi_mention_state) : 0);
  const size_t o_sum = n * sizeof(oi_mention_state), out_bytes = o_sum + n * sizeof(oi_social_summary);
  const uint32_t grid = n_terms < (1u << 20) ? n_terms : (1u << 20);
  auto launch = [&](const unsigned char *d_in, unsigned char *d_out) {
    mention_summary_kernel<<<grid, 128, 0, st>>>(h->d_sig_pol, h->d_sig_flags, term_off, oi_bm25_doc_ids(h),
                                                 reinterpret_cast<const uint32_t *>(d_in), n_terms, source, bull_bear_threshold,
                                                 carry_in ? reinterpret_cast<const oi_mention_state *>(d_in + o_carry) : nullptr,
                                                 reinterpret_cast<oi_mention_state *>(d_out),
                                                 reinterpret_cast<oi_social_summary *>(d_out + o_sum));
    ++h->launches;
    return cudaGetLastError();
  };
  if (!h->no_pinned_staging && in_bytes <= OI_PIN_BYTES && out_bytes <= OI_PIN_BYTES) {  // one pinned copy each way
    SlotLease lease(h, lock);
    oi_index::Slot *sl = lease.sl;
    memcpy(sl->h_in, terms, n * sizeof(uint32_t));
    if (carry_in) memcpy(sl->h_in + o_carry, carry_in, n * sizeof(oi_mention_state));
    MN_CK(cudaMemcpyAsync(sl->d_in, sl->h_in, in_bytes, cudaMemcpyHostToDevice, st));
    MN_CK(launch(sl->d_in, sl->d_out));
    MN_CK(cudaMemcpyAsync(sl->h_out, sl->d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    oi_status s = lease.finish(st);
    if (s) return s;
    if (out_state) memcpy(out_state, sl->h_out, n * sizeof(oi_mention_state));
    memcpy(out_summary, sl->h_out + o_sum, n * sizeof(oi_social_summary));
    return OI_OK;
  }
  // a large call: the handle's own device buffers, direct copies from / to the caller's memory
  const size_t o_out = align16(in_bytes);
  if (o_out + out_bytes > h->mention_io_bytes) {
    MN_CK(cudaStreamSynchronize(st));
    cudaFree(h->d_mention_io);
    h->d_mention_io = nullptr;
    h->mention_io_bytes = 0;
    const size_t want = (o_out + out_bytes) + (o_out + out_bytes) / 4;
    MN_CK(cudaMalloc(&h->d_mention_io, want));
    h->mention_io_bytes = want;
  }
  unsigned char *d_in = h->d_mention_io, *d_out = h->d_mention_io + o_out;
  MN_CK(cudaMemcpyAsync(d_in, terms, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  if (carry_in) MN_CK(cudaMemcpyAsync(d_in + o_carry, carry_in, n * sizeof(oi_mention_state), cudaMemcpyHostToDevice, st));
  MN_CK(launch(d_in, d_out));
  if (out_state) MN_CK(cudaMemcpyAsync(out_state, d_out, n * sizeof(oi_mention_state), cudaMemcpyDeviceToHost, st));
  MN_CK(cudaMemcpyAsync(out_summary, d_out + o_sum, n * sizeof(oi_social_summary), cudaMemcpyDeviceToHost, st));
  MN_CK(call_end(h, st));
  MN_CK(cudaStreamSynchronize(st));
  return OI_OK;
}
#undef MN_CK
