// oi_summary.cuh — the reference's social summary (SpeculationEngine::social_summary,
// src/domain/engine/speculation_engine.rs:76-84) as the body of one CTA of 128 threads.  Shared by the lexicon call
// (lexicon.cu: the batch's own signals, post i = element i) and the per-term mention summaries (mention.cu: element i =
// post doc_ids[lo + i] of a posting list).
//
// The mean is a SEQUENTIAL f64 sum in the reference, so it is one here: every partial sum is rounded as the reference
// rounds it and the result is bit-identical.  All threads stream the signals tile by tile into a double-buffered
// shared-memory ring (coalesced; through the index array when there is one) and count the classes (order-free,
// integer); thread 0 runs the add chain over the tile loaded one step earlier, so the chain never waits for memory -- its
// price is the dependent DADD latency (~19 cycles measured) per post with a non-zero polarity, nothing else.  Posts with
// polarity 0 stay out of the chain: s + 0.0 == s exactly, because no signal is -0.0.
#pragma once
#include "internal.h"

constexpr int kSumTile = 2048;

// kIndexed = false: element i is post i, no source filter, no per-source counts, no carry (the lexicon call).
// kIndexed = true: element i is post doc_ids[lo + i]; flags[p] = speculative (bit 0) | source << 1; a post of another
// source than `source` (>= 0) is neither counted nor chained.  The state starts from *carry (NULL = empty) and the
// running state after these posts goes to *out_state (NULL = not wanted); *out is the summary of that state.
// Called by all 128 threads of the CTA; a CTA may call it again for another list.
template <bool kIndexed>
__device__ __forceinline__ void oi_social_summary_cta(const double *polarity, const uint8_t *flags, const uint32_t *doc_ids,
                                                      unsigned long long lo, unsigned long long n, int source, double thr,
                                                      const oi_mention_state *carry, oi_mention_state *out_state,
                                                      oi_social_summary *out) {
  __shared__ double s_v[2][kSumTile];  // the tile's NON-ZERO polarities of counted posts, in post order
  __shared__ int s_m[2];               // how many
  __shared__ int s_wsum[4];
  __shared__ unsigned long long s_cnt[4 + OI_N_SOURCES];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  __syncthreads();  // thread 0 of a previous call is done with s_cnt
  if (tid < 4 + OI_N_SOURCES) s_cnt[tid] = 0ull;
  unsigned long long bullish = 0, bearish = 0, neutral = 0, spec = 0, by_src[OI_N_SOURCES] = {};
  double sum = carry ? carry->sum : 0.0;
  const unsigned long long n_tiles = (n + kSumTile - 1) / kSumTile;
  for (unsigned long long t = 0; t <= n_tiles; ++t) {
    if (t < n_tiles) {  // stage tile t: thread i owns elements 16 i .. 16 i + 15 of the tile
      const unsigned long long base = t * kSumTile + 16ull * tid;
      double v[16];
      int c = 0;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const unsigned long long g = base + j;
        v[j] = 0.0;
        if (g < n) {
          const unsigned long long p = kIndexed ? (unsigned long long)doc_ids[lo + g] : g;
          const double x = polarity[p];
          const uint32_t f = flags[p];
          if (!kIndexed || source < 0 || (int)(f >> 1) == source) {
            v[j] = x;
            if (x > thr) ++bullish;
            else if (x < -thr) ++bearish;
            else ++neutral;
            spec += f & 1u;
            if (kIndexed) {
#pragma unroll
              for (int s = 0; s < OI_N_SOURCES; ++s) by_src[s] += (f >> 1) == (uint32_t)s;
            }
          }
        }
        c += v[j] != 0.0;
      }
      int x = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int y = __shfl_up_sync(0xFFFFFFFFu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) s_wsum[warp] = x;
      __syncthreads();
      int off = x - c;
      for (int w = 0; w < warp; ++w) off += s_wsum[w];
      double *dst = s_v[t & 1];
#pragma unroll
      for (int j = 0; j < 16; ++j)
        if (v[j] != 0.0) dst[off++] = v[j];
      if (tid == 127) s_m[t & 1] = off;
    }
    if (tid == 0 && t > 0) {  // the add chain over tile t - 1, in post order
      const int m = s_m[(t - 1) & 1];
      const double *v = s_v[(t - 1) & 1];
#pragma unroll 8
      for (int i = 0; i < m; ++i) sum += v[i];
    }
    __syncthreads();
  }
  atomicAdd(&s_cnt[0], bullish); atomicAdd(&s_cnt[1], bearish); atomicAdd(&s_cnt[2], neutral); atomicAdd(&s_cnt[3], spec);
  if (kIndexed) {
#pragma unroll
    for (int s = 0; s < OI_N_SOURCES; ++s) atomicAdd(&s_cnt[4 + s], by_src[s]);
  }
  __syncthreads();
  if (tid != 0) return;
  oi_mention_state st = {};
  if (carry) st = *carry;
  st.bullish += s_cnt[0]; st.bearish += s_cnt[1]; st.neutral += s_cnt[2]; st.speculative += s_cnt[3];
  st.total += s_cnt[0] + s_cnt[1] + s_cnt[2];
  if (kIndexed) {
#pragma unroll
    for (int s = 0; s < OI_N_SOURCES; ++s) st.by_source[s] += s_cnt[4 + s];
  }
  st.sum = sum;
  if (out_state) *out_state = st;
  const unsigned long long cnt = st.total;
  double net = cnt == 0 ? 0.0 : st.sum / (double)cnt;
  double si = cnt == 0 ? 0.0 : (double)st.speculative / (double)cnt;
  net = net > 1.0 ? 1.0 : (net < -1.0 ? -1.0 : net);
  si = si > 1.0 ? 1.0 : (si < 0.0 ? 0.0 : si);
  out->total = cnt; out->bullish = st.bullish; out->bearish = st.bearish; out->neutral = st.neutral;
  out->net_sentiment = net; out->speculation_index = si;
  out->bull_bear_ratio = st.bearish == 0 ? -1.0 : (double)st.bullish / (double)st.bearish;
}
