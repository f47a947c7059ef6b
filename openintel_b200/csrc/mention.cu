// mention.cu — per-term social summaries over the BM25 posting lists (docs/SPEC.md §8a).
//
// A post mentions term t iff one of its tokens equals t: the posts that mention t are t's posting list, doc ids
// ascending.  The handle keeps one lexicon signal per post next to the BM25 part (polarity f64, speculative | source << 1
// in a byte), and one launch runs the shared summary body (oi_summary.cuh) once per requested term, one CTA each, over
// the signals gathered through the term's doc ids.  Every term's chain runs next to the others, so a batch costs about
// its longest list's chain (one dependent DADD per mentioning post with a non-zero polarity); the gather hides behind the
// chain in the tile ring.  The running state in and out lets the shards of a document-sharded index continue one
// another's sequential sum in rank order (a relay), which keeps the mean bit-identical to the unsharded one.
//
// Timelines (SPEC §8b): with a creation time per post, a time bucket splits a posting list into doc-order subsequences.
// One thread per requested posting keys it by (term, bucket); one stable radix sort groups the keys, which keeps every
// (term, bucket) segment in doc order because the input is in (term, doc) order; a binary search in the sorted keys gives
// the segment offsets, and the same summary body runs once per segment.  The chains of all segments run side by side,
// so a call costs about its largest segment's chain, plus a fixed cost per segment that dominates when there are
// millions of tiny ones (DESIGN §4.4).
//
// Co-mentions (SPEC §8d): the posts of up to 64 anchors' lists inside a window are marked in a per-post u64 mask (bit i
// = anchor i).  One pass over all postings, the one of the mention counts, then counts for every term the marked posts
// of its list; and the marked postings of the pairs' term lists, kept in (pair, doc) order by a stable selection, are
// the segments the timeline's summary kernel runs over.
//
// Author runs (SPEC §8e): with an author id per post, each requested posting inside a window is keyed by (term, author)
// in a u64; one stable radix sort and a run-length encoding give the (term, author) runs and their post counts, and one
// pass over the sorted postings, balanced over postings rather than runs, adds the runs' integer fields with atomics.
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_run_length_encode.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <cstring>
#include <vector>

#include "handle.h"
#include "oi_postings.cuh"
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

// ---- timelines (SPEC §8b)
// len[i] = the length of term i's list, len[n] = 0: the exclusive scan in place makes len the lists' starts in the
// concatenation of the requested lists and len[n] their total
__global__ void timeline_lengths_kernel(const u64 *term_off, const uint32_t *terms, uint32_t n, u64 *len) {
  for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i <= n; i += (u64)gridDim.x * blockDim.x)
    len[i] = i < n ? term_off[terms[i] + 1] - term_off[terms[i]] : 0;
}

// posting p of the concatenation -> key i * nb + b (term i, bucket b) or the sentinel n * nb when the post's time is
// outside [edges[0], edges[nb]); value = the doc id.  start[0 .. n]: the lists' starts, start[n] = total.  The edges
// are staged in dynamic shared memory when they fit (oi_stage_edges; the launch sizes it).
__global__ void __launch_bounds__(256) timeline_keys_kernel(const u64 *term_off, const uint32_t *doc_ids, const int64_t *times,
                                                            const uint32_t *terms, const u64 *start, uint32_t n, u64 total,
                                                            const int64_t *edges, uint32_t nb, uint32_t *keys, uint32_t *vals) {
  const int64_t *E = oi_stage_edges(edges, nb);
  for (u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x; p < total; p += (u64)gridDim.x * blockDim.x) {
    uint32_t a = 0, b = n;  // the term: start[a] <= p < start[b] (an empty list shares its start with the next one)
    while (b - a > 1) {
      const uint32_t m = (a + b) >> 1;
      if (start[m] <= p) a = m; else b = m;
    }
    const uint32_t doc = doc_ids[term_off[terms[a]] + (p - start[a])];
    const uint32_t bk = oi_time_bucket(E, nb, times[doc]);
    keys[p] = (uint32_t)(bk < nb ? (u64)a * nb + bk : (u64)n * nb);
    vals[p] = doc;
  }
}

// seg_off[j] = the first place of the sorted keys holding a key >= j, j = 0 .. n_seg: segment j is
// [seg_off[j], seg_off[j + 1]), and the sentinel's postings follow seg_off[n_seg]
__global__ void timeline_segments_kernel(const uint32_t *keys, u64 total, u64 n_seg, u64 *seg_off) {
  for (u64 j = blockIdx.x * (u64)blockDim.x + threadIdx.x; j <= n_seg; j += (u64)gridDim.x * blockDim.x) {
    u64 lo = 0, hi = total;
    while (lo < hi) {
      const u64 m = (lo + hi) >> 1;
      if (keys[m] < j) lo = m + 1; else hi = m;
    }
    seg_off[j] = lo;
  }
}

// the summary body, unchanged, once per (term, bucket) segment of the sorted doc ids
__global__ void __launch_bounds__(128) mention_timeline_kernel(const double *polarity, const uint8_t *flags, const uint32_t *docs,
                                                               const u64 *seg_off, u64 n_seg, int source, double thr,
                                                               const oi_mention_state *carry, oi_mention_state *out_state,
                                                               oi_social_summary *out) {
  for (u64 j = blockIdx.x; j < n_seg; j += gridDim.x)
    oi_social_summary_cta<true>(polarity, flags, docs, seg_off[j], seg_off[j + 1] - seg_off[j], source, thr,
                                carry ? carry + j : nullptr, out_state + j, out + j);
}

// ---- mention counts (SPEC §8c)
// One pass over all postings of the shard, load-balanced over the postings: each warp walks tiles of 256 postings
// (oi_postings.cuh), finds each posting's term and its post's bucket, and counts it in counts[term * nb + bucket].  The
// lanes of a warp that hit the same slot -- the common case inside a long list -- add their popcount with one atomic,
// so a head term does not serialise on its few counters.  The doc ids are streamed; the times (and the flags with a
// source filter) are gathered.  Integer counts: any schedule gives the same result.  The edges are staged as in
// timeline_keys_kernel.
__global__ void __launch_bounds__(256) mention_counts_kernel(const u64 *__restrict__ term_off, const uint32_t *__restrict__ doc_ids,
                                                             const int64_t *__restrict__ times, const uint8_t *__restrict__ flags,
                                                             uint32_t n_terms, u64 n_postings, const int64_t *edges, uint32_t nb,
                                                             int source, uint32_t *counts) {
  const int64_t *E = oi_stage_edges(edges, nb);
  const int lane = threadIdx.x & 31;
  const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 tile = warp * OI_BM25_TILE; tile < n_postings; tile += n_warps * OI_BM25_TILE) {
    const TileTerms tt = bm25_tile_terms(term_off, n_terms, tile, n_postings, lane);
    uint32_t lo = tt.lo;
    for (uint32_t u = 0; u < OI_BM25_TILE / 32; ++u) {
      if (tile + 32u * u >= n_postings) break;  // warp-uniform: the whole warp stays in for the match below
      const u64 p = tile + 32u * u + (uint32_t)lane;
      u64 slot = ~0ull;  // no slot: past the end, another source, or outside the edges
      if (p < n_postings) {
        lo = bm25_term_of(term_off, lo, tt.hi, p);
        const uint32_t doc = __ldcs(doc_ids + p);
        if (source < 0 || (flags[doc] >> 1) == source) {
          const uint32_t bk = oi_time_bucket(E, nb, times[doc]);
          if (bk < nb) slot = (u64)lo * nb + bk;
        }
      }
      const uint32_t peers = __match_any_sync(0xFFFFFFFFu, slot);
      if (slot != ~0ull && lane == __ffs(peers) - 1) atomicAdd(counts + slot, (uint32_t)__popc(peers));
    }
  }
}

// ---- co-mentions (SPEC §8d)
// One thread per posting of the requested anchor lists (start[0 .. n]: their starts in the concatenation, start[n] =
// total, read here so the host does not wait for it): a post of anchor i's list inside [since, until) and of the source
// gets bit i of mask[doc].  The window is applied here, so the passes that read the mask read no times.
__global__ void __launch_bounds__(256) comention_mark_kernel(const u64 *term_off, const uint32_t *doc_ids, const int64_t *times,
                                                             const uint8_t *flags, const uint32_t *anchors, const u64 *start,
                                                             uint32_t n, int64_t since, int64_t until, int source, u64 *mask) {
  const u64 total = start[n];
  for (u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x; p < total; p += (u64)gridDim.x * blockDim.x) {
    uint32_t a = 0, b = n;  // the anchor: start[a] <= p < start[b], as in timeline_keys_kernel
    while (b - a > 1) {
      const uint32_t m = (a + b) >> 1;
      if (start[m] <= p) a = m; else b = m;
    }
    const uint32_t doc = doc_ids[term_off[anchors[a]] + (p - start[a])];
    const int64_t t = times[doc];
    if (t >= since && t < until && (source < 0 || (flags[doc] >> 1) == source)) atomicOr(mask + doc, 1ull << a);
  }
}

// One pass over all postings of the shard with the tile walk of mention_counts_kernel: counts[i * n_terms + t] gets
// the postings of term t whose post carries bit i of the mask.  The doc ids are streamed and the mask gathered.  The
// lanes that share the term and the mask word -- the intersection of two matches -- add their popcount with one atomic
// per set bit, so a head term does not serialise on its counters; a warp whose 32 posts carry no bit does no match.
__global__ void __launch_bounds__(256) comention_counts_kernel(const u64 *__restrict__ term_off, const uint32_t *__restrict__ doc_ids,
                                                               const u64 *__restrict__ mask, uint32_t n_terms, u64 n_postings,
                                                               uint32_t *counts) {
  const int lane = threadIdx.x & 31;
  const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 tile = warp * OI_BM25_TILE; tile < n_postings; tile += n_warps * OI_BM25_TILE) {
    const TileTerms tt = bm25_tile_terms(term_off, n_terms, tile, n_postings, lane);
    uint32_t lo = tt.lo;
    for (uint32_t u = 0; u < OI_BM25_TILE / 32; ++u) {
      if (tile + 32u * u >= n_postings) break;  // warp-uniform: the whole warp stays in for the matches below
      const u64 p = tile + 32u * u + (uint32_t)lane;
      u64 m = 0;  // no bit: past the end, or a post no anchor marked
      if (p < n_postings) {
        lo = bm25_term_of(term_off, lo, tt.hi, p);
        m = mask[__ldcs(doc_ids + p)];
      }
      if (!__any_sync(0xFFFFFFFFu, m != 0)) continue;
      const uint32_t peers = __match_any_sync(0xFFFFFFFFu, lo) & __match_any_sync(0xFFFFFFFFu, m);
      if (m && lane == __ffs(peers) - 1) {
        const uint32_t c = (uint32_t)__popc(peers);
        for (u64 r = m; r; r &= r - 1) atomicAdd(counts + (u64)(__ffsll((long long)r) - 1) * n_terms + lo, c);
      }
    }
  }
}

// posting p of the concatenated pair lists (start[0 .. n], start[n] = total) -> key j (pair j), value = the doc id,
// keep = whether the post carries the mask bit anchor_bit[j] of the pair's anchor
__global__ void __launch_bounds__(256) comention_pair_keys_kernel(const u64 *term_off, const uint32_t *doc_ids, const u64 *mask,
                                                                  const uint32_t *terms, const uint32_t *anchor_bit,
                                                                  const u64 *start, uint32_t n, u64 total, uint32_t *keys,
                                                                  uint32_t *vals, uint8_t *keep) {
  for (u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x; p < total; p += (u64)gridDim.x * blockDim.x) {
    uint32_t a = 0, b = n;
    while (b - a > 1) {
      const uint32_t m = (a + b) >> 1;
      if (start[m] <= p) a = m; else b = m;
    }
    const uint32_t doc = doc_ids[term_off[terms[a]] + (p - start[a])];
    keys[p] = a;
    vals[p] = doc;
    keep[p] = (uint8_t)((mask[doc] >> anchor_bit[a]) & 1u);
  }
}

// ---- author runs (SPEC §8e)
// posting p of the concatenated lists (start[0 .. n], start[n] = total) -> key i * n_authors + author[doc] (term i), or
// the sentinel n * n_authors for a post outside [since, until) or of another source; value = the doc id
__global__ void __launch_bounds__(256) author_keys_kernel(const u64 *term_off, const uint32_t *doc_ids, const int64_t *times,
                                                          const uint8_t *flags, const uint32_t *author, const uint32_t *terms,
                                                          const u64 *start, uint32_t n, u64 total, int64_t since,
                                                          int64_t until, int source, u64 n_authors, u64 *keys, uint32_t *vals) {
  for (u64 p = blockIdx.x * (u64)blockDim.x + threadIdx.x; p < total; p += (u64)gridDim.x * blockDim.x) {
    uint32_t a = 0, b = n;  // the term: start[a] <= p < start[b], as in timeline_keys_kernel
    while (b - a > 1) {
      const uint32_t m = (a + b) >> 1;
      if (start[m] <= p) a = m; else b = m;
    }
    const uint32_t doc = doc_ids[term_off[terms[a]] + (p - start[a])];
    const int64_t t = times[doc];
    const bool in = t >= since && t < until && (source < 0 || (flags[doc] >> 1) == source);
    keys[p] = in ? (u64)a * n_authors + author[doc] : (u64)n * n_authors;
    vals[p] = doc;
  }
}

// term_runs[i] = the first of the n_unique sorted run keys that is >= i * n_authors, i = 0 .. n: term i's runs are
// [term_runs[i], term_runs[i + 1]), and term_runs[n] -- the sentinel's place -- is the number of runs without the
// sentinel's
__global__ void author_term_runs_kernel(const u64 *unique, const int *n_unique, uint32_t n, u64 n_authors, u64 *term_runs) {
  for (u64 i = blockIdx.x * (u64)blockDim.x + threadIdx.x; i <= n; i += (u64)gridDim.x * blockDim.x) {
    u64 lo = 0, hi = (u64)*n_unique;
    const u64 want = i * n_authors;
    while (lo < hi) {
      const u64 m = (lo + hi) >> 1;
      if (unique[m] < want) lo = m + 1; else hi = m;
    }
    term_runs[i] = lo;
  }
}

// run r: its term and author from its key, its post count from the run length, and the neutral elements of the sums,
// the min and the max that author_aggregate_kernel fills
__global__ void author_runs_init_kernel(const u64 *unique, const uint32_t *lengths, u64 n_runs, u64 n_authors,
                                        oi_author_run *runs) {
  for (u64 r = blockIdx.x * (u64)blockDim.x + threadIdx.x; r < n_runs; r += (u64)gridDim.x * blockDim.x) {
    const u64 term = unique[r] / n_authors;
    oi_author_run x;
    x.term = (uint32_t)term;
    x.author = (uint32_t)(unique[r] - term * n_authors);
    x.posts = lengths[r];
    x.bullish = x.bearish = x.speculative = x.engagement = 0;
    x.first_at = INT64_MAX;
    x.last_at = INT64_MIN;
    runs[r] = x;
  }
}

// One pass over the sorted postings, load-balanced over the postings rather than the runs: one author with tens of
// thousands of posts is spread over many warps.  A warp takes 32 consecutive postings; the lanes of one run are
// contiguous because the keys are sorted, so __match_any_sync finds them and a segmented shuffle reduction over
// [leader, last] gives their engagement sum and time range.  The leader finds its run among the unique keys and adds
// the popcounts of its peers' bullish / bearish / speculative votes, the sum and the range with one integer atomic
// each.  The sentinel's postings sort last, so a warp that meets only them is done.
__global__ void __launch_bounds__(256) author_aggregate_kernel(const u64 *__restrict__ keys, const uint32_t *__restrict__ docs,
                                                               u64 total, u64 sentinel, const u64 *__restrict__ unique, u64 n_runs,
                                                               const double *__restrict__ polarity, const uint8_t *__restrict__ flags,
                                                               const int64_t *__restrict__ times,
                                                               const uint32_t *__restrict__ engagement, double thr,
                                                               oi_author_run *runs) {
  const int lane = threadIdx.x & 31;
  const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 base = warp * 32; base < total; base += n_warps * 32) {
    const u64 p = base + (uint32_t)lane;
    const u64 key = p < total ? __ldcs(keys + p) : sentinel;
    const bool on = key < sentinel;
    if (!__any_sync(0xFFFFFFFFu, on)) break;  // warp-uniform: every later posting is the sentinel's too
    bool bull = false, bear = false, spec = false;
    u64 eng = 0;
    int64_t t_lo = INT64_MAX, t_hi = INT64_MIN;
    if (on) {
      const uint32_t doc = __ldcs(docs + p);
      const double x = polarity[doc];
      bull = x > thr;
      bear = x < -thr;
      spec = flags[doc] & 1u;
      eng = engagement[doc];
      t_lo = t_hi = times[doc];
    }
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, on ? key : ~0ull);
    const int last = 31 - __clz(peers);
    for (int o = 1; o < 32; o <<= 1) {  // lane l ends with [l, min(l + 31, last)]: the leader with its whole segment
      const u64 e2 = __shfl_down_sync(0xFFFFFFFFu, eng, o);
      const int64_t lo2 = __shfl_down_sync(0xFFFFFFFFu, t_lo, o), hi2 = __shfl_down_sync(0xFFFFFFFFu, t_hi, o);
      if (lane + o <= last) {
        eng += e2;
        t_lo = lo2 < t_lo ? lo2 : t_lo;
        t_hi = hi2 > t_hi ? hi2 : t_hi;
      }
    }
    const uint32_t b_bull = __ballot_sync(0xFFFFFFFFu, bull), b_bear = __ballot_sync(0xFFFFFFFFu, bear);
    const uint32_t b_spec = __ballot_sync(0xFFFFFFFFu, spec);
    if (on && lane == __ffs(peers) - 1) {
      u64 lo = 0, hi = n_runs;  // the run: unique[lo] == key
      while (lo < hi) {
        const u64 m = (lo + hi) >> 1;
        if (unique[m] < key) lo = m + 1; else hi = m;
      }
      oi_author_run *r = runs + lo;
      if (const uint32_t c = __popc(b_bull & peers)) atomicAdd(reinterpret_cast<unsigned long long *>(&r->bullish), (u64)c);
      if (const uint32_t c = __popc(b_bear & peers)) atomicAdd(reinterpret_cast<unsigned long long *>(&r->bearish), (u64)c);
      if (const uint32_t c = __popc(b_spec & peers)) atomicAdd(reinterpret_cast<unsigned long long *>(&r->speculative), (u64)c);
      if (eng) atomicAdd(reinterpret_cast<unsigned long long *>(&r->engagement), eng);
      atomicMin(reinterpret_cast<long long *>(&r->first_at), (long long)t_lo);
      atomicMax(reinterpret_cast<long long *>(&r->last_at), (long long)t_hi);
    }
  }
}

size_t align16(size_t x) { return (x + 15) & ~(size_t)15; }

// the dynamic shared memory of a kernel that stages nb + 1 edges (oi_stage_edges)
size_t edges_smem(uint32_t nb) { return nb < kEdgesInSmem ? ((size_t)nb + 1) * sizeof(int64_t) : 0; }

// a grow-on-demand device buffer of the handle: at least `want` bytes, with 25 % headroom when it grows
cudaError_t grow(unsigned char *&buf, size_t &cap, size_t want, cudaStream_t st) {
  if (want <= cap) return cudaSuccess;
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) return e;
  cudaFree(buf);
  buf = nullptr;
  cap = 0;
  e = cudaMalloc(&buf, want + want / 4);
  if (e == cudaSuccess) cap = want + want / 4;
  return e;
}

// What a mention call takes: term ids (summary, timeline, co-mentions, authors), bucket edges and the post times
// (timeline, counts, co-mentions and authors: their window is one bucket), the messages of its NULL-argument and
// no-bucket refusals, the name of its term ids in a refusal (nullptr: "terms"), and the post authors (author runs).
struct MentionCall {
  bool terms, edges;
  const char *null_args, *no_bucket, *ids;
  bool authors;
};
constexpr MentionCall kSummary{true, false, "NULL terms / out_summary", nullptr};
constexpr MentionCall kTimeline{true, true, "NULL terms / edges / out_summary", "n_buckets = 0: a timeline needs a bucket"};
constexpr MentionCall kCounts{false, true, "NULL edges / out_counts", "n_buckets = 0: counts need a bucket"};
constexpr MentionCall kComentionCounts{true, true, "NULL anchors / window / out_counts", nullptr, "anchors"};
constexpr MentionCall kComentionPairs{true, true, "NULL anchor_terms / terms / window / out_summary", nullptr, "terms"};
constexpr MentionCall kAuthors{true, true, "NULL terms / window / out_term_runs / out_runs / out_n_runs", nullptr, "terms", true};

// The state and argument checks of the mention calls, in the order they find a fault: the BM25 part, the signals, the
// times and the authors; no term (OI_OK, nothing to do -- with any pointers); a NULL argument, no bucket, more (term, bucket)
// segments than 32-bit keys hold, edges that do not increase strictly, the source, the term ids.  Under the lock.
oi_status mention_check(oi_index *h, const MentionCall &c, const uint32_t *terms, uint32_t n_terms, const int64_t *edges,
                        uint32_t n_buckets, int32_t source, const void *out) {
  if (!oi_bm25_term_offsets(h)) return h->fail(OI_ERR_STATE, "no BM25 part: the posting lists are the mentions");
  if (!h->has_signals) return h->fail(OI_ERR_STATE, "no post signals loaded (oi_index_load_post_signals)");
  if (c.edges && !h->has_times) return h->fail(OI_ERR_STATE, "no post times loaded (oi_index_load_post_times)");
  if (c.authors && !h->has_authors) return h->fail(OI_ERR_STATE, "no post authors loaded (oi_index_load_post_authors)");
  if (c.terms && n_terms == 0) return OI_OK;
  if ((c.terms && !terms) || (c.edges && !edges) || !out) return h->fail(OI_ERR_INVALID_ARG, "%s", c.null_args);
  if (c.edges && n_buckets == 0) return h->fail(OI_ERR_INVALID_ARG, "%s", c.no_bucket);
  const u64 n_seg = (u64)n_terms * n_buckets;
  if (c.terms && c.edges && n_seg > 0xFFFFFFFFull)  // the keys are u32 and the sentinel is n_seg itself
    return h->fail(OI_ERR_INVALID_ARG, "n_terms x n_buckets = %llu: at most 2^32 - 1", (unsigned long long)n_seg);
  if (c.edges)
    for (uint32_t b = 0; b < n_buckets; ++b)
      if (!(edges[b] < edges[b + 1]))
        return h->fail(OI_ERR_INVALID_ARG, "edges[%u] = %lld, edges[%u] = %lld: the edges must increase strictly", b,
                       (long long)edges[b], b + 1, (long long)edges[b + 1]);
  if (source < -1 || source >= OI_N_SOURCES)
    return h->fail(OI_ERR_INVALID_ARG, "source = %d: -1 (all posts) or a source code below %d", source, OI_N_SOURCES);
  const uint32_t V = oi_bm25_n_terms(h);
  if (c.terms)
    for (uint32_t i = 0; i < n_terms; ++i)
      if (terms[i] >= V)
        return h->fail(OI_ERR_INVALID_ARG, "%s[%u] = %u: the BM25 part has %u terms", c.ids ? c.ids : "terms", i, terms[i], V);
  return OI_OK;
}

// the mask of the co-mention calls: clear it, then bit i of mask[doc] for every post of anchors[i]'s list in [since,
// until) and of the source.  d_anchors: n <= 64 term ids on the device; d_start: n + 1 u64 for their lists' starts;
// scan_tmp: the scan's temporaries (scan_bytes of them).
cudaError_t comention_mark(oi_index *h, cudaStream_t st, const uint32_t *d_anchors, uint32_t n, u64 *d_start, void *scan_tmp,
                           size_t scan_bytes, const int64_t *window, int32_t source, u64 *d_mask) {
  const u64 *term_off = oi_bm25_term_offsets(h);
  cudaError_t e = cudaMemsetAsync(d_mask, 0, (h->desc.n_docs ? h->desc.n_docs : 1) * sizeof(u64), st);
  if (e != cudaSuccess) return e;
  timeline_lengths_kernel<<<oi_grid(n + 1, 256, h->num_sms), 256, 0, st>>>(term_off, d_anchors, n, d_start);
  ++h->launches;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = cub::DeviceScan::ExclusiveSum(scan_tmp, scan_bytes, d_start, d_start, (int64_t)n + 1, st)) != cudaSuccess) return e;
  h->launches += 2;
  // the anchors' postings are not known on the host: a resident grid strides over them
  comention_mark_kernel<<<4 * h->num_sms, 256, 0, st>>>(term_off, oi_bm25_doc_ids(h), h->d_times, h->d_sig_flags, d_anchors,
                                                        d_start, n, window[0], window[1], source, d_mask);
  ++h->launches;
  return cudaGetLastError();
}

}  // namespace

void oi_mention_free(oi_index *h) {
  cudaFree(h->d_sig_pol);
  cudaFree(h->d_sig_flags);
  cudaFree(h->d_mention_io);
  cudaFree(h->d_times);
  cudaFree(h->d_timeline_ws);
  h->d_sig_pol = nullptr;
  h->d_sig_flags = nullptr;
  h->d_mention_io = nullptr;
  h->mention_io_bytes = 0;
  h->has_signals = false;
  h->d_times = nullptr;
  h->has_times = false;
  h->d_timeline_ws = nullptr;
  h->timeline_ws_bytes = 0;
  cudaFree(h->d_author);
  cudaFree(h->d_engagement);
  h->d_author = nullptr;
  h->d_engagement = nullptr;
  h->n_authors = 0;
  h->has_authors = false;
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
  OI_CK(cudaSetDevice(h->desc.device));
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
  OI_CK(call_begin(h, h->stream));
  h->has_signals = false;  // until the copies have landed
  if (n) {
    OI_CK(cudaMemcpyAsync(h->d_sig_pol, pol.data(), n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    OI_CK(cudaMemcpyAsync(h->d_sig_flags, fl.data(), n, cudaMemcpyHostToDevice, h->stream));
  }
  OI_CK(call_end(h, h->stream));
  OI_CK(cudaStreamSynchronize(h->stream));
  h->has_signals = true;
  return OI_OK;
}

extern "C" oi_status oi_index_mention_summary(oi_index *h, const uint32_t *terms, uint32_t n_terms, int32_t source,
                                              double bull_bear_threshold, const oi_mention_state *carry_in,
                                              oi_mention_state *out_state, oi_social_summary *out_summary) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::unique_lock<std::mutex> lock(h->mu);
  const oi_status s = mention_check(h, kSummary, terms, n_terms, nullptr, 0, source, out_summary);
  if (s || n_terms == 0) return s;
  const u64 *term_off = oi_bm25_term_offsets(h);
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));
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
    OI_CK(cudaMemcpyAsync(sl->d_in, sl->h_in, in_bytes, cudaMemcpyHostToDevice, st));
    OI_CK(launch(sl->d_in, sl->d_out));
    OI_CK(cudaMemcpyAsync(sl->h_out, sl->d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    if (oi_status f = lease.finish(st)) return f;
    if (out_state) memcpy(out_state, sl->h_out, n * sizeof(oi_mention_state));
    memcpy(out_summary, sl->h_out + o_sum, n * sizeof(oi_social_summary));
    return OI_OK;
  }
  // a large call: the handle's own device buffers, direct copies from / to the caller's memory
  const size_t o_out = align16(in_bytes);
  OI_CK(grow(h->d_mention_io, h->mention_io_bytes, o_out + out_bytes, st));
  unsigned char *d_in = h->d_mention_io, *d_out = h->d_mention_io + o_out;
  OI_CK(cudaMemcpyAsync(d_in, terms, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  if (carry_in) OI_CK(cudaMemcpyAsync(d_in + o_carry, carry_in, n * sizeof(oi_mention_state), cudaMemcpyHostToDevice, st));
  OI_CK(launch(d_in, d_out));
  if (out_state) OI_CK(cudaMemcpyAsync(out_state, d_out, n * sizeof(oi_mention_state), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_summary, d_out + o_sum, n * sizeof(oi_social_summary), cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

extern "C" oi_status oi_index_load_post_times(oi_index *h, const int64_t *created_at) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  if (!created_at) return h->fail(OI_ERR_INVALID_ARG, "NULL created_at");
  const u64 n = h->desc.n_docs;
  OI_CK(cudaSetDevice(h->desc.device));
  if (!h->d_times) {
    const cudaError_t e = cudaMalloc(&h->d_times, (n ? n : 1) * sizeof(int64_t));
    if (e != cudaSuccess) {
      h->d_times = nullptr;
      return h->fail(e == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, "allocating the post times failed: %s",
                     cudaGetErrorString(e));
    }
  }
  OI_CK(call_begin(h, h->stream));
  h->has_times = false;  // until the copy has landed
  if (n) OI_CK(cudaMemcpyAsync(h->d_times, created_at, n * sizeof(int64_t), cudaMemcpyHostToDevice, h->stream));
  OI_CK(call_end(h, h->stream));
  OI_CK(cudaStreamSynchronize(h->stream));
  h->has_times = true;
  return OI_OK;
}

extern "C" oi_status oi_index_mention_timeline(oi_index *h, const uint32_t *terms, uint32_t n_terms, const int64_t *edges,
                                               uint32_t n_buckets, int32_t source, double bull_bear_threshold,
                                               const oi_mention_state *carry_in, oi_mention_state *out_state,
                                               oi_social_summary *out_summary) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  const oi_status s = mention_check(h, kTimeline, terms, n_terms, edges, n_buckets, source, out_summary);
  if (s || n_terms == 0) return s;
  const u64 *term_off = oi_bm25_term_offsets(h);
  const u64 n_seg = (u64)n_terms * n_buckets;
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));

  // d_mention_io: terms u32 [n] | edges i64 [B + 1] | starts u64 [n + 1] | carries [n B] (when given) | states [n B] |
  // summaries [n B] | scan temporaries
  const size_t n = n_terms, nb = n_buckets;
  size_t scan_tmp = 0;
  OI_CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (u64 *)nullptr, (u64 *)nullptr, (int64_t)n + 1, st));
  const size_t o_edges = align16(n * sizeof(uint32_t)), o_start = align16(o_edges + (nb + 1) * sizeof(int64_t));
  const size_t o_carry = align16(o_start + (n + 1) * sizeof(u64));
  const size_t o_state = align16(o_carry + (carry_in ? n_seg * sizeof(oi_mention_state) : 0));
  const size_t o_sum = align16(o_state + n_seg * sizeof(oi_mention_state));
  const size_t o_tmp = align16(o_sum + n_seg * sizeof(oi_social_summary));
  OI_CK(grow(h->d_mention_io, h->mention_io_bytes, o_tmp + scan_tmp, st));
  unsigned char *io = h->d_mention_io;
  uint32_t *d_terms = reinterpret_cast<uint32_t *>(io);
  int64_t *d_edges = reinterpret_cast<int64_t *>(io + o_edges);
  u64 *d_start = reinterpret_cast<u64 *>(io + o_start);
  oi_mention_state *d_carry = carry_in ? reinterpret_cast<oi_mention_state *>(io + o_carry) : nullptr;
  oi_mention_state *d_state = reinterpret_cast<oi_mention_state *>(io + o_state);
  oi_social_summary *d_sum = reinterpret_cast<oi_social_summary *>(io + o_sum);
  OI_CK(cudaMemcpyAsync(d_terms, terms, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  OI_CK(cudaMemcpyAsync(d_edges, edges, (nb + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  if (carry_in) OI_CK(cudaMemcpyAsync(d_carry, carry_in, n_seg * sizeof(oi_mention_state), cudaMemcpyHostToDevice, st));
  timeline_lengths_kernel<<<oi_grid(n + 1, 256, h->num_sms), 256, 0, st>>>(term_off, d_terms, n_terms, d_start);
  ++h->launches;
  OI_CK(cudaGetLastError());
  OI_CK(cub::DeviceScan::ExclusiveSum(io + o_tmp, scan_tmp, d_start, d_start, (int64_t)n + 1, st));
  h->launches += 2;
  u64 total = 0;
  OI_CK(cudaMemcpyAsync(&total, d_start + n, sizeof(u64), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaStreamSynchronize(st));

  // d_timeline_ws: keys u32 [P] x 2 | doc ids u32 [P] x 2 | segment offsets u64 [n B + 1] | sort temporaries
  int end_bit = 0;
  while (end_bit < 32 && (n_seg >> end_bit)) ++end_bit;  // the bits of the largest key, the sentinel n B
  size_t sort_tmp = 0;
  if (total) {
    cub::DoubleBuffer<uint32_t> kb(nullptr, nullptr), vb(nullptr, nullptr);
    OI_CK(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, kb, vb, (int64_t)total, 0, end_bit, st));
  }
  const size_t o_seg = align16(4 * total * sizeof(uint32_t)), o_stmp = align16(o_seg + (n_seg + 1) * sizeof(u64));
  OI_CK(grow(h->d_timeline_ws, h->timeline_ws_bytes, o_stmp + sort_tmp, st));
  unsigned char *ws = h->d_timeline_ws;
  uint32_t *d_keys = reinterpret_cast<uint32_t *>(ws);
  u64 *d_seg = reinterpret_cast<u64 *>(ws + o_seg);
  const uint32_t *sorted_keys = d_keys, *sorted_docs = nullptr;
  if (total) {
    timeline_keys_kernel<<<oi_grid(total, 256, h->num_sms), 256, edges_smem(n_buckets), st>>>(
        term_off, oi_bm25_doc_ids(h), h->d_times, d_terms, d_start, n_terms, total, d_edges, n_buckets, d_keys, d_keys + 2 * total);
    ++h->launches;
    OI_CK(cudaGetLastError());
    // stable: the input is in (term, doc) order, so every (term, bucket) segment stays in doc order
    cub::DoubleBuffer<uint32_t> kb(d_keys, d_keys + total), vb(d_keys + 2 * total, d_keys + 3 * total);
    OI_CK(cub::DeviceRadixSort::SortPairs(ws + o_stmp, sort_tmp, kb, vb, (int64_t)total, 0, end_bit, st));
    h->launches += 1 + (end_bit + 7) / 8;  // histogram + one pass per 8 bits
    sorted_keys = kb.Current();
    sorted_docs = vb.Current();
  }
  timeline_segments_kernel<<<oi_grid(n_seg + 1, 256, h->num_sms), 256, 0, st>>>(sorted_keys, total, n_seg, d_seg);
  ++h->launches;
  OI_CK(cudaGetLastError());
  // a grid that stays resident walks the segments: most are tiny, so no CTA is launched for a single one of them
  int per_sm = 0;
  OI_CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mention_timeline_kernel, 128, 0));
  const u64 resident = (u64)h->num_sms * (u64)(per_sm > 0 ? per_sm : 1);
  mention_timeline_kernel<<<(unsigned)(n_seg < resident ? n_seg : resident), 128, 0, st>>>(
      h->d_sig_pol, h->d_sig_flags, sorted_docs, d_seg, n_seg, source, bull_bear_threshold, d_carry, d_state, d_sum);
  ++h->launches;
  OI_CK(cudaGetLastError());
  if (out_state) OI_CK(cudaMemcpyAsync(out_state, d_state, n_seg * sizeof(oi_mention_state), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_summary, d_sum, n_seg * sizeof(oi_social_summary), cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

extern "C" oi_status oi_index_mention_counts(oi_index *h, const int64_t *edges, uint32_t n_buckets, int32_t source,
                                             uint32_t *out_counts) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  const oi_status s = mention_check(h, kCounts, nullptr, 0, edges, n_buckets, source, out_counts);
  if (s) return s;
  const u64 *term_off = oi_bm25_term_offsets(h);
  const uint32_t V = oi_bm25_n_terms(h);
  const u64 n_seg = (u64)V * n_buckets, nb1 = (u64)n_buckets + 1;
  if (n_seg == 0) return OI_OK;
  // d_mention_io: edges i64 [B + 1] | counts u32 [V B]; the byte count cannot wrap below 2^64
  if (n_seg > (~(u64)0 - 64 - nb1 * sizeof(int64_t)) / sizeof(uint32_t))
    return h->fail(OI_ERR_OUT_OF_MEMORY, "%u terms x %u buckets of counts do not fit the address space", V, n_buckets);
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));
  const size_t o_counts = align16(nb1 * sizeof(int64_t)), bytes = n_seg * sizeof(uint32_t);
  OI_CK(grow(h->d_mention_io, h->mention_io_bytes, o_counts + bytes, st));
  int64_t *d_edges = reinterpret_cast<int64_t *>(h->d_mention_io);
  uint32_t *d_counts = reinterpret_cast<uint32_t *>(h->d_mention_io + o_counts);
  OI_CK(cudaMemsetAsync(d_counts, 0, bytes, st));
  const u64 P = oi_bm25_n_postings(h);
  if (P) {  // a shard without a posting (the token-free shard of a sharded lift) counts nothing
    OI_CK(cudaMemcpyAsync(d_edges, edges, nb1 * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    const size_t smem = edges_smem(n_buckets);
    int per_sm = 0;
    OI_CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mention_counts_kernel, 256, smem));
    const u64 tiles = (P + OI_BM25_TILE - 1) / OI_BM25_TILE, want = (tiles + 7) / 8;  // 8 warps per CTA
    const u64 resident = (u64)h->num_sms * (u64)(per_sm > 0 ? per_sm : 1);
    mention_counts_kernel<<<(unsigned)(want < resident ? want : resident), 256, smem, st>>>(
        term_off, oi_bm25_doc_ids(h), h->d_times, h->d_sig_flags, V, P, d_edges, n_buckets, source, d_counts);
    ++h->launches;
    OI_CK(cudaGetLastError());
  }
  OI_CK(cudaMemcpyAsync(out_counts, d_counts, bytes, cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

extern "C" oi_status oi_index_comention_counts(oi_index *h, const uint32_t *anchors, uint32_t n_anchors, const int64_t *window,
                                               int32_t source, uint32_t *out_counts) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  const oi_status s = mention_check(h, kComentionCounts, anchors, n_anchors, window, 1, source, out_counts);
  if (s || n_anchors == 0) return s;
  if (n_anchors > OI_MAX_COMENTION_ANCHORS)
    return h->fail(OI_ERR_INVALID_ARG, "n_anchors = %u: at most %d anchors, one mask bit each", n_anchors, OI_MAX_COMENTION_ANCHORS);
  const uint32_t V = oi_bm25_n_terms(h);
  const u64 n_out = (u64)n_anchors * V, na1 = (u64)n_anchors + 1;
  // d_mention_io: anchors u32 [64] | starts u64 [65] | counts u32 [n V] | scan temporaries; the byte count cannot wrap
  size_t scan_tmp = 0;
  OI_CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (u64 *)nullptr, (u64 *)nullptr, (int64_t)na1, h->stream));
  const size_t o_start = align16(OI_MAX_COMENTION_ANCHORS * sizeof(uint32_t));
  const size_t o_counts = align16(o_start + (OI_MAX_COMENTION_ANCHORS + 1) * sizeof(u64));
  if (n_out > (~(u64)0 - 64 - o_counts - scan_tmp) / sizeof(uint32_t))
    return h->fail(OI_ERR_OUT_OF_MEMORY, "%u anchors x %u terms of counts do not fit the address space", n_anchors, V);
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));
  const size_t bytes = n_out * sizeof(uint32_t), o_tmp = align16(o_counts + bytes);
  OI_CK(grow(h->d_mention_io, h->mention_io_bytes, o_tmp + scan_tmp, st));
  unsigned char *io = h->d_mention_io;
  uint32_t *d_anchors = reinterpret_cast<uint32_t *>(io), *d_counts = reinterpret_cast<uint32_t *>(io + o_counts);
  OI_CK(cudaMemsetAsync(d_counts, 0, bytes, st));
  const u64 P = oi_bm25_n_postings(h);
  if (P) {  // a shard without a posting (the token-free shard of a sharded lift) counts nothing
    // d_timeline_ws: the mask u64 [n_docs]
    OI_CK(grow(h->d_timeline_ws, h->timeline_ws_bytes, (h->desc.n_docs ? h->desc.n_docs : 1) * sizeof(u64), st));
    u64 *d_mask = reinterpret_cast<u64 *>(h->d_timeline_ws);
    OI_CK(cudaMemcpyAsync(d_anchors, anchors, n_anchors * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    OI_CK(comention_mark(h, st, d_anchors, n_anchors, reinterpret_cast<u64 *>(io + o_start), io + o_tmp, scan_tmp, window,
                         source, d_mask));
    int per_sm = 0;
    OI_CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, comention_counts_kernel, 256, 0));
    const u64 tiles = (P + OI_BM25_TILE - 1) / OI_BM25_TILE, want = (tiles + 7) / 8;  // 8 warps per CTA
    const u64 resident = (u64)h->num_sms * (u64)(per_sm > 0 ? per_sm : 1);
    comention_counts_kernel<<<(unsigned)(want < resident ? want : resident), 256, 0, st>>>(oi_bm25_term_offsets(h), oi_bm25_doc_ids(h),
                                                                                            d_mask, V, P, d_counts);
    ++h->launches;
    OI_CK(cudaGetLastError());
  }
  OI_CK(cudaMemcpyAsync(out_counts, d_counts, bytes, cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

extern "C" oi_status oi_index_comention_summary(oi_index *h, const uint32_t *anchor_terms, const uint32_t *terms, uint32_t n_pairs,
                                                const int64_t *window, int32_t source, double bull_bear_threshold,
                                                const oi_mention_state *carry_in, oi_mention_state *out_state,
                                                oi_social_summary *out_summary) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  // a NULL anchor_terms is refused with the other NULL arguments.  The pairs are keyed by u32 j < n_pairs <= 2^32 - 1.
  const oi_status s = mention_check(h, kComentionPairs, terms, n_pairs, window, 1, source, anchor_terms ? out_summary : nullptr);
  if (s || n_pairs == 0) return s;
  const uint32_t V = oi_bm25_n_terms(h);
  // the distinct anchor terms, first-seen order, and each pair's mask bit: its anchor's place among them
  std::vector<uint32_t> anchors, bit(n_pairs);
  for (uint32_t j = 0; j < n_pairs; ++j) {
    const uint32_t a = anchor_terms[j];
    if (a >= V) return h->fail(OI_ERR_INVALID_ARG, "anchor_terms[%u] = %u: the BM25 part has %u terms", j, a, V);
    uint32_t i = 0;
    while (i < anchors.size() && anchors[i] != a) ++i;
    if (i == anchors.size()) {
      if (i == OI_MAX_COMENTION_ANCHORS)
        return h->fail(OI_ERR_INVALID_ARG, "anchor_terms[%u] = %u: at most %d distinct anchor terms, one mask bit each", j, a,
                       OI_MAX_COMENTION_ANCHORS);
      anchors.push_back(a);
    }
    bit[j] = i;
  }
  const u64 *term_off = oi_bm25_term_offsets(h);
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));

  // d_mention_io: anchors u32 [64] | anchor starts u64 [65] | terms u32 [n] | mask bits u32 [n] | starts u64 [n + 1] |
  // carries [n] (when given) | states [n] | summaries [n] | scan temporaries
  const size_t n = n_pairs, na = anchors.size();
  size_t scan_tmp = 0, scan_a = 0;
  OI_CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (u64 *)nullptr, (u64 *)nullptr, (int64_t)n + 1, st));
  OI_CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_a, (u64 *)nullptr, (u64 *)nullptr, (int64_t)na + 1, st));
  if (scan_a > scan_tmp) scan_tmp = scan_a;
  const size_t o_astart = align16(OI_MAX_COMENTION_ANCHORS * sizeof(uint32_t));
  const size_t o_terms = align16(o_astart + (OI_MAX_COMENTION_ANCHORS + 1) * sizeof(u64));
  const size_t o_bit = align16(o_terms + n * sizeof(uint32_t)), o_start = align16(o_bit + n * sizeof(uint32_t));
  const size_t o_carry = align16(o_start + (n + 1) * sizeof(u64));
  const size_t o_state = align16(o_carry + (carry_in ? n * sizeof(oi_mention_state) : 0));
  const size_t o_sum = align16(o_state + n * sizeof(oi_mention_state));
  const size_t o_tmp = align16(o_sum + n * sizeof(oi_social_summary));
  OI_CK(grow(h->d_mention_io, h->mention_io_bytes, o_tmp + scan_tmp, st));
  unsigned char *io = h->d_mention_io;
  uint32_t *d_anchors = reinterpret_cast<uint32_t *>(io), *d_terms = reinterpret_cast<uint32_t *>(io + o_terms);
  uint32_t *d_bit = reinterpret_cast<uint32_t *>(io + o_bit);
  u64 *d_start = reinterpret_cast<u64 *>(io + o_start);
  oi_mention_state *d_carry = carry_in ? reinterpret_cast<oi_mention_state *>(io + o_carry) : nullptr;
  oi_mention_state *d_state = reinterpret_cast<oi_mention_state *>(io + o_state);
  oi_social_summary *d_sum = reinterpret_cast<oi_social_summary *>(io + o_sum);
  OI_CK(cudaMemcpyAsync(d_anchors, anchors.data(), na * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  OI_CK(cudaMemcpyAsync(d_terms, terms, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  OI_CK(cudaMemcpyAsync(d_bit, bit.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  if (carry_in) OI_CK(cudaMemcpyAsync(d_carry, carry_in, n * sizeof(oi_mention_state), cudaMemcpyHostToDevice, st));
  timeline_lengths_kernel<<<oi_grid(n + 1, 256, h->num_sms), 256, 0, st>>>(term_off, d_terms, n_pairs, d_start);
  ++h->launches;
  OI_CK(cudaGetLastError());
  OI_CK(cub::DeviceScan::ExclusiveSum(io + o_tmp, scan_tmp, d_start, d_start, (int64_t)n + 1, st));
  h->launches += 2;
  u64 total = 0;
  OI_CK(cudaMemcpyAsync(&total, d_start + n, sizeof(u64), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaStreamSynchronize(st));

  // d_timeline_ws: mask u64 [n_docs] | keys u32 [P] | doc ids u32 [P] | kept keys u32 [P] | kept doc ids u32 [P] |
  // keep u8 [P] | kept count i64 | segment offsets u64 [n + 1] | select temporaries
  size_t sel_tmp = 0;
  if (total)
    OI_CK(cub::DeviceSelect::Flagged(nullptr, sel_tmp, (const uint32_t *)nullptr, (const uint8_t *)nullptr, (uint32_t *)nullptr,
                                     (int64_t *)nullptr, (int64_t)total, st));
  const size_t o_keys = align16((h->desc.n_docs ? h->desc.n_docs : 1) * sizeof(u64));
  const size_t o_keep = align16(o_keys + 4 * total * sizeof(uint32_t)), o_nsel = align16(o_keep + total);
  const size_t o_seg = align16(o_nsel + sizeof(int64_t)), o_stmp = align16(o_seg + (n + 1) * sizeof(u64));
  OI_CK(grow(h->d_timeline_ws, h->timeline_ws_bytes, o_stmp + sel_tmp, st));
  unsigned char *ws = h->d_timeline_ws;
  u64 *d_mask = reinterpret_cast<u64 *>(ws), *d_seg = reinterpret_cast<u64 *>(ws + o_seg);
  uint32_t *d_keys = reinterpret_cast<uint32_t *>(ws + o_keys);
  uint32_t *kept_keys = d_keys + 2 * total, *kept_docs = d_keys + 3 * total;
  if (total) {
    OI_CK(comention_mark(h, st, d_anchors, (uint32_t)na, reinterpret_cast<u64 *>(io + o_astart), io + o_tmp, scan_tmp, window,
                         source, d_mask));
    comention_pair_keys_kernel<<<oi_grid(total, 256, h->num_sms), 256, 0, st>>>(
        term_off, oi_bm25_doc_ids(h), d_mask, d_terms, d_bit, d_start, n_pairs, total, d_keys, d_keys + total, ws + o_keep);
    ++h->launches;
    OI_CK(cudaGetLastError());
    // the kept keys past the kept count read 0xFFFFFFFF, above every pair, so the segment search runs over all P of them.
    // Stable: the concatenation is in (pair, doc) order, so each pair's kept posts stay in doc order.
    OI_CK(cudaMemsetAsync(kept_keys, 0xFF, total * sizeof(uint32_t), st));
    int64_t *d_nsel = reinterpret_cast<int64_t *>(ws + o_nsel);
    OI_CK(cub::DeviceSelect::Flagged(ws + o_stmp, sel_tmp, d_keys, ws + o_keep, kept_keys, d_nsel, (int64_t)total, st));
    OI_CK(cub::DeviceSelect::Flagged(ws + o_stmp, sel_tmp, d_keys + total, ws + o_keep, kept_docs, d_nsel, (int64_t)total, st));
    h->launches += 4;  // init + select, twice
  }
  timeline_segments_kernel<<<oi_grid(n + 1, 256, h->num_sms), 256, 0, st>>>(kept_keys, total, n, d_seg);
  ++h->launches;
  OI_CK(cudaGetLastError());
  int per_sm = 0;
  OI_CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mention_timeline_kernel, 128, 0));
  const u64 resident = (u64)h->num_sms * (u64)(per_sm > 0 ? per_sm : 1);
  mention_timeline_kernel<<<(unsigned)(n < resident ? n : resident), 128, 0, st>>>(
      h->d_sig_pol, h->d_sig_flags, total ? kept_docs : nullptr, d_seg, n, source, bull_bear_threshold, d_carry, d_state, d_sum);
  ++h->launches;
  OI_CK(cudaGetLastError());
  if (out_state) OI_CK(cudaMemcpyAsync(out_state, d_state, n * sizeof(oi_mention_state), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaMemcpyAsync(out_summary, d_sum, n * sizeof(oi_social_summary), cudaMemcpyDeviceToHost, st));
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

extern "C" oi_status oi_index_load_post_authors(oi_index *h, const uint32_t *author, const uint32_t *engagement) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  if (!author || !engagement) return h->fail(OI_ERR_INVALID_ARG, "NULL author / engagement");
  const u64 n = h->desc.n_docs;
  uint32_t top = 0;
  for (u64 i = 0; i < n; ++i) top = author[i] > top ? author[i] : top;
  OI_CK(cudaSetDevice(h->desc.device));
  if (!h->d_author) {
    cudaError_t e = cudaMalloc(&h->d_author, (n ? n : 1) * sizeof(uint32_t));
    if (e == cudaSuccess) e = cudaMalloc(&h->d_engagement, (n ? n : 1) * sizeof(uint32_t));
    if (e != cudaSuccess) {
      cudaFree(h->d_author);
      h->d_author = nullptr;
      h->d_engagement = nullptr;
      return h->fail(e == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, "allocating the post authors failed: %s",
                     cudaGetErrorString(e));
    }
  }
  OI_CK(call_begin(h, h->stream));
  h->has_authors = false;  // until the copies have landed
  if (n) {
    OI_CK(cudaMemcpyAsync(h->d_author, author, n * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    OI_CK(cudaMemcpyAsync(h->d_engagement, engagement, n * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  }
  OI_CK(call_end(h, h->stream));
  OI_CK(cudaStreamSynchronize(h->stream));
  h->n_authors = (u64)top + 1;
  h->has_authors = true;
  return OI_OK;
}

extern "C" oi_status oi_index_mention_authors(oi_index *h, const uint32_t *terms, uint32_t n_terms, const int64_t *window,
                                              int32_t source, double bull_bear_threshold, uint64_t capacity,
                                              uint64_t *out_term_runs, oi_author_run *out_runs, uint64_t *out_n_runs) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  const oi_status s = mention_check(h, kAuthors, terms, n_terms, window, 1, source,
                                    out_term_runs && out_runs && out_n_runs ? out_runs : nullptr);
  if (s || n_terms == 0) return s;
  const u64 *term_off = oi_bm25_term_offsets(h);
  const u64 n_authors = h->n_authors, sentinel = (u64)n_terms * n_authors;  // < 2^64: n_terms < 2^32, n_authors <= 2^32
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  OI_CK(call_begin(h, st));

  // d_mention_io: terms u32 [n] | starts u64 [n + 1] | term runs u64 [n + 1] | scan temporaries
  const size_t n = n_terms;
  size_t scan_tmp = 0;
  OI_CK(cub::DeviceScan::ExclusiveSum(nullptr, scan_tmp, (u64 *)nullptr, (u64 *)nullptr, (int64_t)n + 1, st));
  const size_t o_start = align16(n * sizeof(uint32_t)), o_truns = align16(o_start + (n + 1) * sizeof(u64));
  const size_t o_tmp = align16(o_truns + (n + 1) * sizeof(u64));
  OI_CK(grow(h->d_mention_io, h->mention_io_bytes, o_tmp + scan_tmp, st));
  unsigned char *io = h->d_mention_io;
  uint32_t *d_terms = reinterpret_cast<uint32_t *>(io);
  u64 *d_start = reinterpret_cast<u64 *>(io + o_start), *d_truns = reinterpret_cast<u64 *>(io + o_truns);
  OI_CK(cudaMemcpyAsync(d_terms, terms, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  timeline_lengths_kernel<<<oi_grid(n + 1, 256, h->num_sms), 256, 0, st>>>(term_off, d_terms, n_terms, d_start);
  ++h->launches;
  OI_CK(cudaGetLastError());
  OI_CK(cub::DeviceScan::ExclusiveSum(io + o_tmp, scan_tmp, d_start, d_start, (int64_t)n + 1, st));
  h->launches += 2;
  u64 total = 0;
  OI_CK(cudaMemcpyAsync(&total, d_start + n, sizeof(u64), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaStreamSynchronize(st));
  if (total > 0x7FFFFFFFull)  // the run-length encoding counts items in an int
    return h->fail(OI_ERR_INVALID_ARG, "the requested lists hold %llu postings: at most 2^31 - 1 in one call",
                   (unsigned long long)total);

  // d_timeline_ws: keys u64 [P] x 2 | doc ids u32 [P] x 2 | run keys u64 [P] | run lengths u32 [P] | run count i32 |
  // sort / encode temporaries
  int end_bit = 0;
  while (end_bit < 64 && (sentinel >> end_bit)) ++end_bit;  // the bits of the largest key, the sentinel
  size_t sort_tmp = 0, rle_tmp = 0;
  if (total) {
    cub::DoubleBuffer<u64> kb(nullptr, nullptr);
    cub::DoubleBuffer<uint32_t> vb(nullptr, nullptr);
    OI_CK(cub::DeviceRadixSort::SortPairs(nullptr, sort_tmp, kb, vb, (int64_t)total, 0, end_bit, st));
    OI_CK(cub::DeviceRunLengthEncode::Encode(nullptr, rle_tmp, (const u64 *)nullptr, (u64 *)nullptr, (uint32_t *)nullptr,
                                             (int *)nullptr, (int)total, st));
  }
  const size_t o_vals = align16(2 * total * sizeof(u64)), o_uniq = align16(o_vals + 2 * total * sizeof(uint32_t));
  const size_t o_len = align16(o_uniq + total * sizeof(u64)), o_nruns = align16(o_len + total * sizeof(uint32_t));
  const size_t o_wtmp = align16(o_nruns + sizeof(int));
  OI_CK(grow(h->d_timeline_ws, h->timeline_ws_bytes, o_wtmp + (sort_tmp > rle_tmp ? sort_tmp : rle_tmp), st));
  unsigned char *ws = h->d_timeline_ws;
  u64 *d_keys = reinterpret_cast<u64 *>(ws), *d_uniq = reinterpret_cast<u64 *>(ws + o_uniq);
  uint32_t *d_vals = reinterpret_cast<uint32_t *>(ws + o_vals), *d_len = reinterpret_cast<uint32_t *>(ws + o_len);
  int *d_nruns = reinterpret_cast<int *>(ws + o_nruns);
  const u64 *sorted_keys = d_keys;
  const uint32_t *sorted_docs = d_vals;
  if (total) {
    author_keys_kernel<<<oi_grid(total, 256, h->num_sms), 256, 0, st>>>(
        term_off, oi_bm25_doc_ids(h), h->d_times, h->d_sig_flags, h->d_author, d_terms, d_start, n_terms, total, window[0],
        window[1], source, n_authors, d_keys, d_vals);
    ++h->launches;
    OI_CK(cudaGetLastError());
    cub::DoubleBuffer<u64> kb(d_keys, d_keys + total);
    cub::DoubleBuffer<uint32_t> vb(d_vals, d_vals + total);
    OI_CK(cub::DeviceRadixSort::SortPairs(ws + o_wtmp, sort_tmp, kb, vb, (int64_t)total, 0, end_bit, st));
    h->launches += 1 + (end_bit + 7) / 8;  // histogram + one pass per 8 bits
    sorted_keys = kb.Current();
    sorted_docs = vb.Current();
    OI_CK(cub::DeviceRunLengthEncode::Encode(ws + o_wtmp, rle_tmp, sorted_keys, d_uniq, d_len, d_nruns, (int)total, st));
    h->launches += 2;
  } else {
    OI_CK(cudaMemsetAsync(d_nruns, 0, sizeof(int), st));
  }
  author_term_runs_kernel<<<oi_grid(n + 1, 256, h->num_sms), 256, 0, st>>>(d_uniq, d_nruns, n_terms, n_authors, d_truns);
  ++h->launches;
  OI_CK(cudaGetLastError());
  std::vector<u64> term_runs(n + 1);
  OI_CK(cudaMemcpyAsync(term_runs.data(), d_truns, (n + 1) * sizeof(u64), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaStreamSynchronize(st));
  const u64 n_runs = term_runs[n];
  *out_n_runs = n_runs;
  if (n_runs > capacity)
    return h->fail(OI_ERR_INVALID_ARG, "%llu runs do not fit capacity = %llu", (unsigned long long)n_runs,
                   (unsigned long long)capacity);
  if (n_runs) {
    // d_mention_io (its terms and starts are spent): runs [R]
    OI_CK(grow(h->d_mention_io, h->mention_io_bytes, n_runs * sizeof(oi_author_run), st));
    oi_author_run *d_runs = reinterpret_cast<oi_author_run *>(h->d_mention_io);
    author_runs_init_kernel<<<oi_grid(n_runs, 256, h->num_sms), 256, 0, st>>>(d_uniq, d_len, n_runs, n_authors, d_runs);
    ++h->launches;
    OI_CK(cudaGetLastError());
    author_aggregate_kernel<<<oi_grid(total, 256, h->num_sms), 256, 0, st>>>(
        sorted_keys, sorted_docs, total, sentinel, d_uniq, n_runs, h->d_sig_pol, h->d_sig_flags, h->d_times, h->d_engagement,
        bull_bear_threshold, d_runs);
    ++h->launches;
    OI_CK(cudaGetLastError());
    OI_CK(cudaMemcpyAsync(out_runs, d_runs, n_runs * sizeof(oi_author_run), cudaMemcpyDeviceToHost, st));
  }
  OI_CK(call_end(h, st));
  OI_CK(cudaStreamSynchronize(st));
  memcpy(out_term_runs, term_runs.data(), (n + 1) * sizeof(u64));
  return OI_OK;
}
