// oi_postings.cuh — shared device helpers of the per-posting kernels over the BM25 CSR: the term of a posting (the
// warp-tile walk of bm25.cu's weight and validation kernels, also used by mention.cu's counts), and the staged edges
// and the time bucket of a post (mention.cu's timelines and counts, SPEC §8b).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "oi_common.cuh"

// Term of posting p = the last t with term_off[t] <= p, searched inside [lo, hi) (invariant: term_off[lo] <= p <
// term_off[hi]).  The per-posting kernels walk the postings in warp tiles of 256: two full searches per tile (its
// first and last posting) bound every other search to the few terms the tile spans -- none at all in the long lists.
__device__ __forceinline__ uint32_t bm25_term_of(const u64 *__restrict__ term_off, uint32_t lo, uint32_t hi, u64 p) {
  while (hi - lo > 1) {
    const uint32_t mid = lo + ((hi - lo) >> 1);
    if (__ldg(term_off + mid) <= p) lo = mid; else hi = mid;
  }
  return lo;
}
#define OI_BM25_TILE 256u
struct TileTerms { uint32_t lo, hi; };
__device__ __forceinline__ TileTerms bm25_tile_terms(const u64 *__restrict__ term_off, uint32_t n_terms, u64 tile, u64 n_postings, int lane) {
  const u64 last = min(tile + OI_BM25_TILE - 1, n_postings - 1);
  uint32_t b = 0;
  if (lane == 0) b = bm25_term_of(term_off, 0, n_terms, tile);
  if (lane == 31) b = bm25_term_of(term_off, 0, n_terms, last);
  TileTerms t;
  t.lo = __shfl_sync(0xFFFFFFFFu, b, 0);
  t.hi = __shfl_sync(0xFFFFFFFFu, b, 31) + 1;
  return t;
}

// The edges E[0 .. nb] of a bucketed kernel, staged in the block's dynamic shared memory when nb < kEdgesInSmem (the
// launch gives (nb + 1) * 8 bytes then, else none) and read from global memory otherwise.  Every thread of the block
// calls it; -> the edges the block reads.
constexpr int kEdgesInSmem = 4096;
__device__ __forceinline__ const int64_t *oi_stage_edges(const int64_t *edges, uint32_t nb) {
  extern __shared__ int64_t s_dyn_edges[];
  const bool staged = nb < kEdgesInSmem;
  if (staged)
    for (uint32_t k = threadIdx.x; k <= nb; k += blockDim.x) s_dyn_edges[k] = edges[k];
  __syncthreads();
  return staged ? s_dyn_edges : edges;
}

// The bucket of time t among the strictly increasing edges E[0 .. nb]: b with E[b] <= t < E[b + 1], or nb when t is
// outside [E[0], E[nb]) (SPEC §8b).
__device__ __forceinline__ uint32_t oi_time_bucket(const int64_t *E, uint32_t nb, int64_t t) {
  if (!(t >= E[0] && t < E[nb])) return nb;
  uint32_t lo = 0, hi = nb;
  while (hi - lo > 1) {
    const uint32_t m = (lo + hi) >> 1;
    if (E[m] <= t) lo = m; else hi = m;
  }
  return lo;
}
