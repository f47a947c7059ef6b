// cosine_scan.cu — single-query cosine scan over the resident embedding matrix with the top-k
// fused in (scores never reach HBM).  Bandwidth-bound GEMV: SURVEY.md §8d config 2.
//
//   algorithmic bytes per query = n_rows * dim * sizeof(T)        (roofline numerator)
//
// Two variants of the same contract:
//   0  cosine_scan_ldg_kernel   one warp per row group, 128-bit ld.global.nc.L1::no_allocate,
//                               ROWS x NVL independent loads in flight per lane, 2 CTAs / SM.
//   1  cosine_scan_bulk_kernel  one producer warp streams row tiles with cp.async.bulk
//                               (TMA 1-D, SASS UBLKCP) through an mbarrier ring in shared
//                               memory; 8 consumer warps reduce rows from shared memory.
// Both: warp-shuffle reduction per row, 64-bit (score, doc) keys (SPEC §1), a per-CTA candidate
// buffer filtered by a running threshold (oi_common.cuh), a grid-wide threshold exchanged with
// atomicMax, and a last-CTA merge of the per-CTA lists — one launch per query, no second kernel.
#include <cuda_bf16.h>

#include "internal.h"
#include "oi_common.cuh"

static int g_tile_rows_override = 0, g_stages_override = 0;  // tuning experiments (oi_index_set_option)
void oi_cosine_scan_tuning(int tile_rows, int stages) { g_tile_rows_override = tile_rows; g_stages_override = stages; }

namespace {

constexpr int kConsumerThreads = 256;
constexpr int kConsumerWarps = kConsumerThreads / 32;

// ---- element traits: a 16-byte vector holds QF elements ----------------------------------------
template <typename T>
struct Elem;
template <>
struct Elem<float> {
  static constexpr int QF = 4;
  __device__ static __forceinline__ void load_q(const float *q, uint32_t v, float *out) {
    float4 t = *reinterpret_cast<const float4 *>(q + (size_t)v * 4);
    out[0] = t.x; out[1] = t.y; out[2] = t.z; out[3] = t.w;
  }
  __device__ static __forceinline__ float dot(uint4 d, const float *q, float acc) {
    acc = fmaf(__uint_as_float(d.x), q[0], acc);
    acc = fmaf(__uint_as_float(d.y), q[1], acc);
    acc = fmaf(__uint_as_float(d.z), q[2], acc);
    acc = fmaf(__uint_as_float(d.w), q[3], acc);
    return acc;
  }
};
template <>
struct Elem<__nv_bfloat16> {
  static constexpr int QF = 8;
  // SPEC §2 bf16 path: the query is rounded to bf16 (RNE) once, then used as f32
  __device__ static __forceinline__ void load_q(const float *q, uint32_t v, float *out) {
    float4 a = *reinterpret_cast<const float4 *>(q + (size_t)v * 8);
    float4 b = *reinterpret_cast<const float4 *>(q + (size_t)v * 8 + 4);
    float t[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
    for (int i = 0; i < 8; ++i) out[i] = __bfloat162float(__float2bfloat16_rn(t[i]));
  }
  __device__ static __forceinline__ float dot(uint4 d, const float *q, float acc) {
    acc = fmaf(__uint_as_float(d.x << 16), q[0], acc);
    acc = fmaf(__uint_as_float(d.x & 0xFFFF0000u), q[1], acc);
    acc = fmaf(__uint_as_float(d.y << 16), q[2], acc);
    acc = fmaf(__uint_as_float(d.y & 0xFFFF0000u), q[3], acc);
    acc = fmaf(__uint_as_float(d.z << 16), q[4], acc);
    acc = fmaf(__uint_as_float(d.z & 0xFFFF0000u), q[5], acc);
    acc = fmaf(__uint_as_float(d.w << 16), q[6], acc);
    acc = fmaf(__uint_as_float(d.w & 0xFFFF0000u), q[7], acc);
    return acc;
  }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
  return v;
}

__device__ __forceinline__ u64 ld_relaxed_u64(const u64 *p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// ---- shared selection state of one CTA --------------------------------------------------------
struct SelState {
  u64 buf[OI_SEL_CAP];
  u64 thr;
  uint32_t cnt;
  uint32_t is_last;
};

// Exact top-k of G sorted (descending, 0-padded) lists of k keys, list c at lists + c * stride.  On return
// S.buf[0 .. S.cnt) holds the result, sorted.  Called by the `nthreads` threads of barrier `bar`.
//  (1) sampling bound: if m lists each hold >= ceil(k/m) keys >= T then at least k keys are >= T;
//  (2) every list is sorted, so its keys above the bound are a prefix: measure the prefixes (gallop + bisect,
//      ~3 dependent loads per list) and, when they fit the buffer together — the common case, a few hundred
//      keys — copy them in place; otherwise (heavy ties, skewed lists, G > OI_SEL_CAP) stream every key
//      through the filter + buffer.  One CTA does this per query, so it has to take microseconds.
//  `known` (0 = none) is a key the caller knows at least k keys of the lists reach (the BM25 kernel's running
//  threshold): it replaces the sampling bound when it is the stronger one.
__device__ void merge_sorted_lists(SelState &S, const u64 *lists, uint32_t G, size_t stride, uint32_t k, int tid, int nthreads, int bar,
                                   u64 known = 0ull) {
  bool fits = false;
  if (tid == 0) { S.cnt = 0; S.thr = 0ull; }
  oi_bar_sync(bar, nthreads);
  if (G <= OI_SEL_CAP / 2) {  // G sample keys below, 2 G prefix words above the middle of the buffer
    const uint32_t m = max(1u, G / 2);
    const uint32_t j = (k + m - 1) / m - 1;
    const uint32_t gp = oi_next_pow2(G);
    for (uint32_t c = tid; c < gp; c += nthreads) S.buf[c] = c < G ? __ldcg(lists + (size_t)c * stride + j) : 0ull;
    oi_bar_sync(bar, nthreads);
    oi_bitonic_desc(S.buf, gp, tid, nthreads, bar);
    const u64 T = S.buf[m - 1];
    oi_bar_sync(bar, nthreads);
    const u64 bound = max(T > 0 ? T - 1 : 0ull, known > 0 ? known - 1 : 0ull);
    uint32_t *s_n = reinterpret_cast<uint32_t *>(S.buf + OI_SEL_CAP / 2);  // [G] prefix lengths, then [G] offsets
    uint32_t *s_off = s_n + G;
    for (uint32_t c = tid; c < G; c += nthreads) {
      const u64 *list = lists + (size_t)c * stride;
      uint32_t lo = 0, hi = 1;  // keys [0, lo) pass; find the first position that does not
      while (hi <= k && __ldcg(list + hi - 1) > bound) { lo = hi; hi <<= 1; }
      hi = min(hi - 1, k);      // position hi (if < k) fails or is the end
      while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldcg(list + mid) > bound) lo = mid + 1; else hi = mid;
      }
      s_n[c] = lo;
    }
    oi_bar_sync(bar, nthreads);
    if (tid == 0) {
      uint32_t sum = 0;
      for (uint32_t c = 0; c < G; ++c) { s_off[c] = sum; sum += s_n[c]; }
      S.is_last = sum;  // broadcast slot for the total
    }
    oi_bar_sync(bar, nthreads);
    const uint32_t total_pass = S.is_last;
    fits = total_pass <= OI_SEL_CAP / 2;
    if (fits) {
      for (uint32_t c = tid; c < G; c += nthreads) {
        const u64 *list = lists + (size_t)c * stride;
        const uint32_t n = s_n[c], o = s_off[c];
        for (uint32_t i = 0; i < n; ++i) S.buf[o + i] = __ldcg(list + i);
      }
      oi_bar_sync(bar, nthreads);
      if (tid == 0) S.cnt = total_pass;
      oi_bar_sync(bar, nthreads);
      oi_sel_compact(S.buf, &S.cnt, &S.thr, k, tid, nthreads, bar);
    } else {
      if (tid == 0) S.thr = bound;
      oi_bar_sync(bar, nthreads);
    }
  }
  if (!fits) {
    const u64 total = (u64)G * k;
    u64 base = 0;
    while (base < total) {
      // snapshot (cnt, thr) before anybody pushes: loop bounds must be CTA-uniform
      const uint32_t span = (uint32_t)min(total - base, (u64)((uint32_t)OI_SEL_CAP - S.cnt));
      const u64 thr = S.thr;
      oi_bar_sync(bar, nthreads);
      for (u64 i = base + tid; i < base + span; i += nthreads) {
        const u64 key = __ldcg(lists + (i / k) * stride + (i % k));
        if (key > thr) oi_sel_push(S.buf, &S.cnt, key);
      }
      base += span;
      oi_bar_sync(bar, nthreads);
      if (S.cnt > OI_SEL_CAP / 2 || base >= total) oi_sel_compact(S.buf, &S.cnt, &S.thr, k, tid, nthreads, bar);
    }
  }
}

// Ends a scan CTA: final compaction, publish the sorted local list, and — in the last CTA to
// arrive — merge all lists into out_keys.  Called by the `nthreads` threads of barrier `bar`.
__device__ void scan_epilogue(SelState &S, const OiScanParams &p, int tid, int nthreads, int bar) {
  const uint32_t k = p.k;
  oi_sel_compact(S.buf, &S.cnt, &S.thr, k, tid, nthreads, bar);
  if (tid == 0 && S.cnt == k) atomicMax(p.gthr, S.thr);
  u64 *mine = p.cand + (size_t)blockIdx.x * k;
  for (uint32_t i = tid; i < k; i += nthreads) mine[i] = i < S.cnt ? S.buf[i] : 0ull;
  __threadfence();
  oi_bar_sync(bar, nthreads);
  if (tid == 0) {
    uint32_t t = atomicAdd(p.ticket, 1u);
    S.is_last = (t == gridDim.x - 1);
  }
  oi_bar_sync(bar, nthreads);
  if (!S.is_last) return;
  __threadfence();
  // ---- last CTA: exact top-k of the gridDim.x sorted lists -------------------------------------
  merge_sorted_lists(S, p.cand, gridDim.x, k, k, tid, nthreads, bar);
  // (3) emit and re-arm the per-query control words for the next launch
  for (uint32_t i = tid; i < k; i += nthreads) p.out_keys[i] = i < S.cnt ? S.buf[i] : 0ull;
  if (tid == 0) { *p.ticket = 0; *p.tile_ctr = 0; *p.gthr = 0ull; }
}

// =================================================================================================
// Variant 0: direct loads.  NVL = 16-byte vectors per lane per row (nv <= 32*NVL), ROWS rows in
// flight per warp.
// =================================================================================================
template <typename T, int NVL, int ROWS>
__global__ void __launch_bounds__(kConsumerThreads, 2) cosine_scan_ldg_kernel(const OiScanParams p) {
  constexpr int QF = Elem<T>::QF;
  __shared__ SelState S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

  float q[NVL][QF];
#pragma unroll
  for (int j = 0; j < NVL; ++j) {
    const uint32_t v = lane + 32 * j;
    if (v < p.nv) {
      Elem<T>::load_q(p.q, v, q[j]);
    } else {
#pragma unroll
      for (int e = 0; e < QF; ++e) q[j][e] = 0.0f;
    }
  }
  if (tid == 0) { S.cnt = 0; S.thr = 0ull; }
  __syncthreads();

  const uint32_t row_begin = min(p.n_rows, blockIdx.x * p.rows_per_cta);
  const uint32_t row_end = min(p.n_rows, row_begin + p.rows_per_cta);
  const uint4 *mat = p.mat;
  const uint32_t nv = p.nv;

  uint32_t base = row_begin;
  while (base < row_end) {
    // super-iteration: at most (CAP - cnt) rows, so pushes cannot overflow the buffer
    const uint32_t span = min(row_end - base, (uint32_t)OI_SEL_CAP - S.cnt);
    const u64 thr = max(S.thr, ld_relaxed_u64(p.gthr));
    const uint32_t stop = base + span;
    __syncthreads();  // (cnt, thr) snapshot is CTA-uniform before anybody pushes
    // the loads of the next row pair are in flight while this one is reduced (one pair of look-ahead per warp)
    uint4 dn[ROWS][NVL];
    {
      const uint32_t r0 = base + warp * ROWS;
#pragma unroll
      for (int i = 0; i < ROWS; ++i)
#pragma unroll
        for (int j = 0; j < NVL; ++j) {
          const uint32_t v = lane + 32 * j;
          dn[i][j] = (r0 + i < stop && v < nv) ? oi_ldg_stream(mat + (size_t)(r0 + i) * nv + v) : make_uint4(0, 0, 0, 0);
        }
    }
    for (uint32_t r0 = base + warp * ROWS; r0 < stop; r0 += kConsumerWarps * ROWS) {
      uint4 d[ROWS][NVL];
      const uint32_t rn = r0 + kConsumerWarps * ROWS;
#pragma unroll
      for (int i = 0; i < ROWS; ++i)
#pragma unroll
        for (int j = 0; j < NVL; ++j) {
          const uint32_t v = lane + 32 * j;
          d[i][j] = dn[i][j];
          dn[i][j] = (rn + i < stop && v < nv) ? oi_ldg_stream(mat + (size_t)(rn + i) * nv + v) : make_uint4(0, 0, 0, 0);
        }
      float acc[ROWS];
#pragma unroll
      for (int i = 0; i < ROWS; ++i) {
        float a = 0.0f;
#pragma unroll
        for (int j = 0; j < NVL; ++j) a = Elem<T>::dot(d[i][j], q[j], a);
        acc[i] = warp_sum(a);
      }
      if (lane == 0) {
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
          if (r0 + i < stop) {
            u64 key = oi_make_key(acc[i], p.doc_base + r0 + i);
            if (key > thr) oi_sel_push(S.buf, &S.cnt, key);
          }
        }
      }
    }
    base = stop;
    __syncthreads();
    if (base < row_end && S.cnt > OI_SEL_CAP / 2) {
      oi_sel_compact(S.buf, &S.cnt, &S.thr, p.k, tid, kConsumerThreads, 0);
      if (tid == 0 && S.cnt == p.k) atomicMax(p.gthr, S.thr);
    }
  }
  scan_epilogue(S, p, tid, kConsumerThreads, 0);
}

// =================================================================================================
// Multi-query scan: one pass over the matrix serves a GROUP of up to kMultiQ queries (f32 indexes have no
// tensor-core path -- tf32 products would miss the 1e-5 tolerance -- and bf16 batches below the GEMM threshold
// land here too).  Same structure as variant 0 (direct 128-bit loads, 2 CTAs per SM, contiguous row ranges);
// the group's queries sit in registers, every loaded row vector is used kMultiQ times, and the kMultiQ x 2
// partial sums of a row pair are reduced together: a butterfly that halves the number of live values at each of
// its first three steps (9 shuffles instead of 40).  One selection state per query in dynamic shared memory;
// the per-query epilogue (publish, last-CTA merge) is the single-query one.  The bytes stay the bound: per row
// 3 loads, 48 FMAs and ~5 shuffles per lane at dim 384, ~20 issue cycles per row and SM against ~50 of HBM time.
// =================================================================================================
// Warp reduction of 8 values at once: the first three butterfly steps halve the number of live values (a lane
// keeps the half selected by its bit 4, 3, 2 and sends the other), the last two finish the one that is left:
// 4 + 2 + 1 + 1 + 1 = 9 shuffles instead of 8 x 5.  On return lanes 4i .. 4i+3 hold the full sum of value i.
__device__ __forceinline__ float multi_reduce8(const float (&v8)[8], int lane) {
  float v4[4], v2[2];
  {
    const bool hi = lane & 16;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float send = hi ? v8[j] : v8[j + 4], keep = hi ? v8[j + 4] : v8[j];
      v4[j] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, 16);
    }
  }
  {
    const bool hi = lane & 8;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const float send = hi ? v4[j] : v4[j + 2], keep = hi ? v4[j + 2] : v4[j];
      v2[j] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, 8);
    }
  }
  float v1;
  {
    const bool hi = lane & 4;
    const float send = hi ? v2[0] : v2[1], keep = hi ? v2[1] : v2[0];
    v1 = keep + __shfl_xor_sync(0xFFFFFFFFu, send, 4);
  }
  v1 += __shfl_xor_sync(0xFFFFFFFFu, v1, 2);
  v1 += __shfl_xor_sync(0xFFFFFFFFu, v1, 1);
  return v1;
}

constexpr int kMultiQ = 4;

template <typename T, int NVL>
__global__ void __launch_bounds__(kConsumerThreads, 2) cosine_scan_multi_kernel(const OiScanParams p) {
  constexpr int QF = Elem<T>::QF;
  constexpr int ROWS = 2;
  extern __shared__ __align__(16) unsigned char s_multi[];
  SelState *S = reinterpret_cast<SelState *>(s_multi);  // [kMultiQ]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t ng = p.nq;  // queries in this group, 1..kMultiQ (CTA-uniform)

  float q[kMultiQ][NVL][QF];
#pragma unroll
  for (int g = 0; g < kMultiQ; ++g)
#pragma unroll
    for (int j = 0; j < NVL; ++j) {
      const uint32_t v = lane + 32 * j;
      if ((uint32_t)g < ng && v < p.nv) {
        Elem<T>::load_q(p.q + (size_t)g * p.dim, v, q[g][j]);
      } else {
#pragma unroll
        for (int e = 0; e < QF; ++e) q[g][j][e] = 0.0f;
      }
    }
  if (tid < kMultiQ) { S[tid].cnt = 0; S[tid].thr = 0ull; }
  __syncthreads();

  const uint32_t row_begin = min(p.n_rows, blockIdx.x * p.rows_per_cta);
  const uint32_t row_end = min(p.n_rows, row_begin + p.rows_per_cta);
  const uint4 *mat = p.mat;
  const uint32_t nv = p.nv;
  // after the butterfly, lanes 4i .. 4i+3 hold value i = query (i >> 1), row (i & 1) of the pair
  const int my_val = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
  const int my_g = my_val >> 1, my_i = my_val & 1;

  // The first super-iterations are short (128, 256, 512, ... rows) and a buffer is cut to its best k as soon as it
  // holds 2k keys: the first thresholds then come from sorts of a few hundred keys.  (Scanning 2048 rows without
  // a threshold and sorting 2048 keys per query cost a third of the pass.)
  uint32_t span_cap = 128;
  const uint32_t ctrig = min((uint32_t)OI_SEL_CAP / 2, max(2u * p.k, 128u));
  uint32_t base = row_begin;
  while (base < row_end) {
    // super-iteration: at most (CAP - cnt) rows for the fullest buffer, so pushes cannot overflow any of them
    uint32_t room = span_cap;
    span_cap = min(span_cap * 2, (uint32_t)OI_SEL_CAP);
    for (uint32_t g = 0; g < ng; ++g) room = min(room, (uint32_t)OI_SEL_CAP - S[g].cnt);
    const u64 my_thr = (uint32_t)my_g < ng ? max(S[my_g].thr, ld_relaxed_u64(p.gthr + my_g)) : ~0ull;
    const uint32_t stop = base + min(row_end - base, room);
    __syncthreads();  // (cnt, thr) snapshots are CTA-uniform before anybody pushes
    // the loads of the next row pair are in flight while this one is reduced (one pair of look-ahead per warp)
    uint4 dn[ROWS][NVL];
    {
      const uint32_t r0 = base + warp * ROWS;
#pragma unroll
      for (int i = 0; i < ROWS; ++i)
#pragma unroll
        for (int j = 0; j < NVL; ++j) {
          const uint32_t v = lane + 32 * j;
          dn[i][j] = (r0 + i < stop && v < nv) ? oi_ldg_stream(mat + (size_t)(r0 + i) * nv + v) : make_uint4(0, 0, 0, 0);
        }
    }
    for (uint32_t r0 = base + warp * ROWS; r0 < stop; r0 += kConsumerWarps * ROWS) {
      uint4 d[ROWS][NVL];
      const uint32_t rn = r0 + kConsumerWarps * ROWS;
#pragma unroll
      for (int i = 0; i < ROWS; ++i)
#pragma unroll
        for (int j = 0; j < NVL; ++j) {
          const uint32_t v = lane + 32 * j;
          d[i][j] = dn[i][j];
          dn[i][j] = (rn + i < stop && v < nv) ? oi_ldg_stream(mat + (size_t)(rn + i) * nv + v) : make_uint4(0, 0, 0, 0);
        }
      float v8[kMultiQ * ROWS];
#pragma unroll
      for (int g = 0; g < kMultiQ; ++g)
#pragma unroll
        for (int i = 0; i < ROWS; ++i) {
          float a = 0.0f;
#pragma unroll
          for (int j = 0; j < NVL; ++j) a = Elem<T>::dot(d[i][j], q[g][j], a);
          v8[g * ROWS + i] = a;
        }
      const float v1 = multi_reduce8(v8, lane);
      if ((lane & 3) == 0 && r0 + my_i < stop) {
        const u64 key = oi_make_key(v1, p.doc_base + r0 + my_i);
        if (key > my_thr) oi_sel_push(S[my_g].buf, &S[my_g].cnt, key);
      }
    }
    base = stop;
    __syncthreads();
    if (base < row_end) {
      for (uint32_t g = 0; g < ng; ++g) {
        if (S[g].cnt > ctrig) {  // CTA-uniform: read after the barrier
          oi_sel_compact(S[g].buf, &S[g].cnt, &S[g].thr, p.k, tid, kConsumerThreads, 0);
          if (tid == 0 && S[g].cnt == p.k) atomicMax(p.gthr + g, S[g].thr);
        }
      }
    }
  }
  for (uint32_t g = 0; g < ng; ++g) {
    OiScanParams pq = p;
    pq.cand = p.cand + (size_t)g * p.cand_stride;
    pq.gthr = p.gthr + g;
    pq.ticket = p.ticket + g;
    pq.tile_ctr = p.tile_ctr + g;
    pq.out_keys = p.out_keys + (size_t)g * p.k;
    scan_epilogue(S[g], pq, tid, kConsumerThreads, 0);
    __syncthreads();
  }
}

// Generic fallback for wide rows (nv > 256): the query lives in shared memory as f32.
template <typename T>
__global__ void __launch_bounds__(kConsumerThreads, 2) cosine_scan_generic_kernel(const OiScanParams p) {
  constexpr int QF = Elem<T>::QF;
  extern __shared__ __align__(16) float s_q[];  // nv * QF floats
  __shared__ SelState S;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (uint32_t v = tid; v < p.nv; v += kConsumerThreads) Elem<T>::load_q(p.q, v, s_q + (size_t)v * QF);
  if (tid == 0) { S.cnt = 0; S.thr = 0ull; }
  __syncthreads();
  const uint32_t row_begin = min(p.n_rows, blockIdx.x * p.rows_per_cta);
  const uint32_t row_end = min(p.n_rows, row_begin + p.rows_per_cta);
  uint32_t base = row_begin;
  while (base < row_end) {
    const uint32_t span = min(row_end - base, (uint32_t)OI_SEL_CAP - S.cnt);
    const u64 thr = max(S.thr, ld_relaxed_u64(p.gthr));
    const uint32_t stop = base + span;
    __syncthreads();  // (cnt, thr) snapshot is CTA-uniform before anybody pushes
    for (uint32_t r = base + warp; r < stop; r += kConsumerWarps) {
      const uint4 *rp = p.mat + (size_t)r * p.nv;
      float a0 = 0.0f, a1 = 0.0f;
      uint32_t v = lane;
      for (; v + 32 < p.nv; v += 64) {
        uint4 d0 = oi_ldg_stream(rp + v), d1 = oi_ldg_stream(rp + v + 32);
        a0 = Elem<T>::dot(d0, s_q + (size_t)v * QF, a0);
        a1 = Elem<T>::dot(d1, s_q + (size_t)(v + 32) * QF, a1);
      }
      if (v < p.nv) a0 = Elem<T>::dot(oi_ldg_stream(rp + v), s_q + (size_t)v * QF, a0);
      float s = warp_sum(a0 + a1);
      if (lane == 0) {
        u64 key = oi_make_key(s, p.doc_base + r);
        if (key > thr) oi_sel_push(S.buf, &S.cnt, key);
      }
    }
    base = stop;
    __syncthreads();
    if (base < row_end && S.cnt > OI_SEL_CAP / 2) {
      oi_sel_compact(S.buf, &S.cnt, &S.thr, p.k, tid, kConsumerThreads, 0);
      if (tid == 0 && S.cnt == p.k) atomicMax(p.gthr, S.thr);
    }
  }
  scan_epilogue(S, p, tid, kConsumerThreads, 0);
}

// =================================================================================================
// Variant 1 (default): bulk-async-copy pipeline with dynamic tiles.  One CTA per SM.  Warp 8 is
// the producer: it draws row tiles from a grid-wide atomic counter (one ticket ahead, so the
// round trip to L2 is off the critical path) and streams them with cp.async.bulk (TMA 1-D, SASS
// UBLKCP) through an mbarrier ring; warps 0-7 reduce rows from shared memory.  Dynamic tiles make
// every SM finish within one tile of the others (no tail), and the copy engine keeps
// n_stages x tile_bytes (~190 KB) in flight per SM without spending registers on it.
// Dynamic smem: [n_stages][tile_bytes] row tiles (128 B aligned), 2*n_stages mbarriers, then
// n_stages u32 tile ids.
// =================================================================================================
constexpr uint32_t kTileEnd = 0xFFFFFFFFu;
constexpr int kBulkWarps = 16;                  // consumer warps of the bulk variant
constexpr int kBulkThreads = kBulkWarps * 32;   // + one producer warp + the epilogue warps
constexpr int kEpiWarps = 4;                    // run a query's list merge while the consumers scan the next query
constexpr int kEpiThreads = kEpiWarps * 32;
constexpr int kBulkBlock = kBulkThreads + 32 + kEpiThreads;

template <typename T, int NVL, bool EXACT>
__global__ void __launch_bounds__(kBulkBlock, 1)
    cosine_scan_bulk_kernel(const OiScanParams p, const uint32_t tile_rows, const uint32_t n_stages) {
  constexpr int QF = Elem<T>::QF;
  extern __shared__ __align__(128) unsigned char s_dyn[];
  // two selection states: query i fills slot i & 1 while the epilogue warps finish query i - 1 in the other
  __shared__ SelState S2[2];
  __shared__ u64 s_qdone[2], s_edone[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t row_bytes = p.nv * 16u;
  const uint32_t tile_bytes = tile_rows * row_bytes;
  u64 *full = reinterpret_cast<u64 *>(s_dyn + (size_t)n_stages * tile_bytes);
  u64 *empty = full + n_stages;
  uint32_t *s_tile = reinterpret_cast<uint32_t *>(empty + n_stages);
  const uint32_t n_tiles = (p.n_rows + tile_rows - 1) / tile_rows;

  if (tid == 0) {
    for (uint32_t s = 0; s < n_stages; ++s) { oi_mbar_init(&full[s], 1); oi_mbar_init(&empty[s], kBulkWarps); }
    for (int b = 0; b < 2; ++b) { oi_mbar_init(&s_qdone[b], 1); oi_mbar_init(&s_edone[b], 1); S2[b].cnt = 0; S2[b].thr = 0ull; }
    oi_mbar_fence_init();
  }
  __syncthreads();

  if (warp > kBulkWarps) {
    // ---------------- epilogue warps: publish + (last CTA) merge the lists of query qi -----------------
    const int etid = tid - (kBulkThreads + 32);
    for (uint32_t qi = 0; qi < p.nq; ++qi) {
      const uint32_t slot = qi & 1u, ph = (qi >> 1) & 1u;
      SelState &S = S2[slot];
      OiScanParams pq = p;
      pq.cand = p.cand + (size_t)qi * p.cand_stride;
      pq.gthr = p.gthr + qi;
      pq.ticket = p.ticket + qi;
      pq.tile_ctr = p.tile_ctr + qi;
      pq.out_keys = p.out_keys + (size_t)qi * p.k;
      oi_mbar_wait(&s_qdone[slot], ph);
      scan_epilogue(S, pq, etid, kEpiThreads, 2);
      oi_bar_sync(2, kEpiThreads);
      if (etid == 0) {
        S.cnt = 0; S.thr = 0ull;
        __threadfence_block();
        oi_mbar_arrive(&s_edone[slot]);
      }
    }
    return;
  }

  if (warp == kBulkWarps) {
    // ---------------- producer: one elected lane, all queries of the batch back to back ----------
    if (lane == 0) {
      const u64 policy = oi_policy_evict_first();
      const unsigned char *src = reinterpret_cast<const unsigned char *>(p.mat);
      uint32_t it = 0;
      for (uint32_t qi = 0; qi < p.nq; ++qi) {
        uint32_t *ctr = p.tile_ctr + qi;
        uint32_t t = atomicAdd(ctr, 1u);
        for (;; ++it) {
          const uint32_t s = it % n_stages, ph = (it / n_stages) & 1u;
          const uint32_t t_next = t < n_tiles ? atomicAdd(ctr, 1u) : kTileEnd;  // ticket for the next round
          oi_mbar_wait(&empty[s], ph ^ 1u);
          if (t >= n_tiles) {
            s_tile[s] = kTileEnd;  // end of this query: the consumers run its epilogue
            oi_mbar_arrive(&full[s]);
            ++it;
            break;
          }
          s_tile[s] = t;
          const uint32_t rows = min(tile_rows, p.n_rows - t * tile_rows);
          const uint32_t bytes = rows * row_bytes;
          oi_mbar_expect_tx(&full[s], bytes);
          oi_bulk_g2s(s_dyn + (size_t)s * tile_bytes, src + (size_t)t * tile_bytes, bytes, &full[s], policy);
          t = t_next;
        }
      }
    }
    return;  // the producer warp takes no part in barrier 1 or the epilogues
  }

  // -------------------------------- consumers --------------------------------------------------
  uint32_t it = 0;
  for (uint32_t qi = 0; qi < p.nq; ++qi) {
    const uint32_t slot = qi & 1u;
    SelState &S = S2[slot];
    OiScanParams pq = p;
    pq.q = p.q + (size_t)qi * p.dim;
    pq.gthr = p.gthr + qi;
    // the slot is free once the epilogue of query qi - 2 has re-armed it
    oi_mbar_wait(&s_edone[slot], ((qi >> 1) & 1u) ^ 1u);
    float q[NVL][QF];
#pragma unroll
    for (int j = 0; j < NVL; ++j) {
      const uint32_t v = lane + 32 * j;
      if (EXACT || v < p.nv) {
        Elem<T>::load_q(pq.q, v, q[j]);
      } else {
#pragma unroll
        for (int e = 0; e < QF; ++e) q[j][e] = 0.0f;
      }
    }
    bool done = false;
    while (!done) {
      // super-iteration over as many tiles as the candidate buffer can absorb in the worst case
      const uint32_t tiles_now = max(1u, ((uint32_t)OI_SEL_CAP - S.cnt) / tile_rows);
      const u64 thr = max(S.thr, ld_relaxed_u64(pq.gthr));
      oi_bar_sync(1, kBulkThreads);  // (cnt, thr) snapshot is uniform before anybody pushes
      for (uint32_t n = 0; n < tiles_now; ++n) {
        const uint32_t s = it % n_stages, ph = (it / n_stages) & 1u;
        oi_mbar_wait(&full[s], ph);
        const uint32_t t = s_tile[s];
        ++it;
        if (t == kTileEnd) {  // every consumer warp sees the same sentinel; the slot holds no data
          __syncwarp();
          if (lane == 0) oi_mbar_arrive(&empty[s]);
          done = true;
          break;
        }
        const uint32_t tile_row0 = t * tile_rows;
        const uint32_t rows = min(tile_rows, p.n_rows - tile_row0);
        const unsigned char *tile = s_dyn + (size_t)s * tile_bytes;
        for (uint32_t r = warp * 2; r < rows; r += kBulkWarps * 2) {
          const uint4 *rp0 = reinterpret_cast<const uint4 *>(tile + (size_t)r * row_bytes);
          const bool two = r + 1 < rows;
          const uint4 *rp1 = two ? reinterpret_cast<const uint4 *>(tile + (size_t)(r + 1) * row_bytes) : rp0;
          float a0[NVL], a1[NVL];
#pragma unroll
          for (int j = 0; j < NVL; ++j) {
            const uint32_t v = lane + 32 * j;
            a0[j] = 0.0f; a1[j] = 0.0f;
            if (EXACT || v < p.nv) {
              a0[j] = Elem<T>::dot(rp0[v], q[j], 0.0f);
              a1[j] = Elem<T>::dot(rp1[v], q[j], 0.0f);
            }
          }
          float s0 = a0[0], s1 = a1[0];
#pragma unroll
          for (int j = 1; j < NVL; ++j) { s0 += a0[j]; s1 += a1[j]; }
          // two rows share one butterfly: after the first exchange lanes 0-15 carry row r,
          // lanes 16-31 row r+1
          const bool hi = lane & 16;
          float keep = hi ? s1 : s0;
          keep += __shfl_xor_sync(0xFFFFFFFFu, hi ? s0 : s1, 16);
          keep += __shfl_xor_sync(0xFFFFFFFFu, keep, 8);
          keep += __shfl_xor_sync(0xFFFFFFFFu, keep, 4);
          keep += __shfl_xor_sync(0xFFFFFFFFu, keep, 2);
          keep += __shfl_xor_sync(0xFFFFFFFFu, keep, 1);
          if ((lane & 15) == 0 && (!hi || two)) {
            const u64 key = oi_make_key(keep, p.doc_base + tile_row0 + r + (hi ? 1u : 0u));
            if (key > thr) oi_sel_push(S.buf, &S.cnt, key);
          }
        }
        __syncwarp();
        if (lane == 0) oi_mbar_arrive(&empty[s]);
      }
      oi_bar_sync(1, kBulkThreads);
      if (!done && S.cnt > OI_SEL_CAP / 2) {
        oi_sel_compact(S.buf, &S.cnt, &S.thr, p.k, tid, kBulkThreads, 1);
        if (tid == 0 && S.cnt == p.k) atomicMax(pq.gthr, S.thr);
      }
    }
    // this query is done in this CTA: hand its candidates to the epilogue warps (final compaction, publish, and
    // in the last CTA to arrive the merge of all lists) and start on the next query's tiles right away
    if (tid == 0) {
      __threadfence_block();
      oi_mbar_arrive(&s_qdone[slot]);
    }
  }
}

// =================================================================================================
// Multi-query scan on the bulk-copy pipeline: the producer warp of variant 1 (dynamic tiles, cp.async.bulk ring)
// feeds 16 consumer warps that hold a GROUP of kMultiQ queries in registers; selection states and epilogue as in
// cosine_scan_multi_kernel (no epilogue overlap: the group's queries finish together).  The copy engine keeps the
// ring full whatever the consumers do, which the direct-load version cannot (its loads stop during every sort).
// Dynamic smem: [n_stages][tile_bytes] | full[n_stages], empty[n_stages] | s_tile[n_stages] | SelState[kMultiQ].
// =================================================================================================
constexpr int kBMBlock = kBulkThreads + 32;

template <typename T, int NVL>
__global__ void __launch_bounds__(kBMBlock, 1)
    cosine_scan_bulk_multi_kernel(const OiScanParams p, const uint32_t tile_rows, const uint32_t n_stages) {
  constexpr int QF = Elem<T>::QF;
  extern __shared__ __align__(128) unsigned char s_dyn[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t row_bytes = p.nv * 16u;
  const uint32_t tile_bytes = tile_rows * row_bytes;
  u64 *full = reinterpret_cast<u64 *>(s_dyn + (size_t)n_stages * tile_bytes);
  u64 *empty = full + n_stages;
  uint32_t *s_tile = reinterpret_cast<uint32_t *>(empty + n_stages);
  SelState *S = reinterpret_cast<SelState *>(s_dyn + (((size_t)n_stages * tile_bytes + n_stages * 20u + 15u) & ~(size_t)15));
  const uint32_t n_tiles = (p.n_rows + tile_rows - 1) / tile_rows;
  const uint32_t ng = p.nq;  // queries in this group, 1..kMultiQ

  if (tid == 0) {
    for (uint32_t s = 0; s < n_stages; ++s) { oi_mbar_init(&full[s], 1); oi_mbar_init(&empty[s], kBulkWarps); }
    for (int g = 0; g < kMultiQ; ++g) { S[g].cnt = 0; S[g].thr = 0ull; }
    oi_mbar_fence_init();
  }
  __syncthreads();

  if (warp == kBulkWarps) {
    // ---------------- producer: one elected lane, one pass over the shard's tiles ----------------
    if (lane == 0) {
      const u64 policy = oi_policy_evict_first();
      const unsigned char *src = reinterpret_cast<const unsigned char *>(p.mat);
      uint32_t *ctr = p.tile_ctr;
      uint32_t t = atomicAdd(ctr, 1u);
      for (uint32_t it = 0;; ++it) {
        const uint32_t s = it % n_stages, ph = (it / n_stages) & 1u;
        const uint32_t t_next = t < n_tiles ? atomicAdd(ctr, 1u) : kTileEnd;  // ticket for the next round
        oi_mbar_wait(&empty[s], ph ^ 1u);
        if (t >= n_tiles) {
          s_tile[s] = kTileEnd;
          oi_mbar_arrive(&full[s]);
          break;
        }
        s_tile[s] = t;
        const uint32_t rows = min(tile_rows, p.n_rows - t * tile_rows);
        const uint32_t bytes = rows * row_bytes;
        oi_mbar_expect_tx(&full[s], bytes);
        oi_bulk_g2s(s_dyn + (size_t)s * tile_bytes, src + (size_t)t * tile_bytes, bytes, &full[s], policy);
        t = t_next;
      }
    }
    return;  // the producer warp takes no part in barrier 1 or the epilogues
  }

  // -------------------------------- consumers --------------------------------------------------
  float q[kMultiQ][NVL][QF];
#pragma unroll
  for (int g = 0; g < kMultiQ; ++g)
#pragma unroll
    for (int j = 0; j < NVL; ++j) {
      const uint32_t v = lane + 32 * j;
      if ((uint32_t)g < ng && v < p.nv) {
        Elem<T>::load_q(p.q + (size_t)g * p.dim, v, q[g][j]);
      } else {
#pragma unroll
        for (int e = 0; e < QF; ++e) q[g][j][e] = 0.0f;
      }
    }
  const int my_val = ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1);
  const int my_g = my_val >> 1, my_i = my_val & 1;
  const uint32_t ctrig = min((uint32_t)OI_SEL_CAP / 2, max(2u * p.k, 128u));
  const uint32_t max_tiles = max(1u, (uint32_t)OI_SEL_CAP / tile_rows);
  uint32_t tiles_cap = max(1u, 128u / tile_rows);  // short first super-iterations: early, cheap thresholds
  uint32_t s = 0, ph = 0;  // ring position (no division per tile)
  bool done = false;
  while (!done) {
    uint32_t room = OI_SEL_CAP;
    for (uint32_t g = 0; g < ng; ++g) room = min(room, (uint32_t)OI_SEL_CAP - S[g].cnt);
    const uint32_t tiles_now = max(1u, min(tiles_cap, room / tile_rows));
    tiles_cap = min(tiles_cap * 2, max_tiles);
    const u64 my_thr = (uint32_t)my_g < ng ? max(S[my_g].thr, ld_relaxed_u64(p.gthr + my_g)) : ~0ull;
    oi_bar_sync(1, kBulkThreads);  // (cnt, thr) snapshots are uniform before anybody pushes
    for (uint32_t n = 0; n < tiles_now; ++n) {
      oi_mbar_wait(&full[s], ph);
      const uint32_t t = s_tile[s];
      const uint32_t s_cur = s;
      if (++s == n_stages) { s = 0; ph ^= 1u; }
      if (t == kTileEnd) {  // every consumer warp sees the same sentinel; the slot holds no data
        __syncwarp();
        if (lane == 0) oi_mbar_arrive(&empty[s_cur]);
        done = true;
        break;
      }
      const uint32_t tile_row0 = t * tile_rows;
      const uint32_t rows = min(tile_rows, p.n_rows - tile_row0);
      const unsigned char *tile = s_dyn + (size_t)s_cur * tile_bytes;
      for (uint32_t r = warp * 2; r < rows; r += kBulkWarps * 2) {
        const uint4 *rp0 = reinterpret_cast<const uint4 *>(tile + (size_t)r * row_bytes);
        const bool two = r + 1 < rows;
        const uint4 *rp1 = two ? reinterpret_cast<const uint4 *>(tile + (size_t)(r + 1) * row_bytes) : rp0;
        uint4 d[2][NVL];
#pragma unroll
        for (int j = 0; j < NVL; ++j) {
          const uint32_t v = lane + 32 * j;
          d[0][j] = v < p.nv ? rp0[v] : make_uint4(0, 0, 0, 0);
          d[1][j] = v < p.nv ? rp1[v] : make_uint4(0, 0, 0, 0);
        }
        float v8[kMultiQ * 2];
#pragma unroll
        for (int g = 0; g < kMultiQ; ++g)
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            float a = 0.0f;
#pragma unroll
            for (int j = 0; j < NVL; ++j) a = Elem<T>::dot(d[i][j], q[g][j], a);
            v8[g * 2 + i] = a;
          }
        const float v1 = multi_reduce8(v8, lane);
        if ((lane & 3) == 0 && (my_i == 0 || two)) {
          const u64 key = oi_make_key(v1, p.doc_base + tile_row0 + r + (uint32_t)my_i);
          if (key > my_thr) oi_sel_push(S[my_g].buf, &S[my_g].cnt, key);
        }
      }
      __syncwarp();
      if (lane == 0) oi_mbar_arrive(&empty[s_cur]);
    }
    oi_bar_sync(1, kBulkThreads);
    if (!done) {
      // warp g cuts query g's buffer to its best k (warp-level sort: the four buffers are compacted at the same
      // time and without CTA barriers)
      if ((uint32_t)warp < ng && S[warp].cnt > ctrig) {
        oi_warp_sel_compact(S[warp].buf, &S[warp].cnt, &S[warp].thr, OI_SEL_CAP, p.k, lane);
        if (lane == 0 && S[warp].cnt == p.k) atomicMax(p.gthr + warp, S[warp].thr);
      }
      // the (cnt, thr) snapshot of the next round is taken before that round's barrier: close this one here
      oi_bar_sync(1, kBulkThreads);
    }
  }
  for (uint32_t g = 0; g < ng; ++g) {
    OiScanParams pq = p;
    pq.cand = p.cand + (size_t)g * p.cand_stride;
    pq.gthr = p.gthr + g;
    pq.ticket = p.ticket + g;
    pq.tile_ctr = p.tile_ctr + g;
    pq.out_keys = p.out_keys + (size_t)g * p.k;
    scan_epilogue(S[g], pq, tid, kBulkThreads, 1);
    oi_bar_sync(1, kBulkThreads);
  }
}

// ---- host-side dispatch -------------------------------------------------------------------------
template <typename T, int NVL, int ROWS>
cudaError_t launch_ldg(const OiScanParams &p, uint32_t grid, cudaStream_t st) {
  cosine_scan_ldg_kernel<T, NVL, ROWS><<<grid, kConsumerThreads, 0, st>>>(p);
  return cudaGetLastError();
}

template <typename T>
cudaError_t dispatch_ldg(const OiScanParams &p, uint32_t grid, cudaStream_t st) {
  const uint32_t nvl = (p.nv + 31) / 32;
  switch (nvl) {
    case 1: return launch_ldg<T, 1, 8>(p, grid, st);
    case 2: return launch_ldg<T, 2, 4>(p, grid, st);
    case 3: return launch_ldg<T, 3, 4>(p, grid, st);
    case 4: return launch_ldg<T, 4, 2>(p, grid, st);
    case 5:
    case 6: return launch_ldg<T, 6, 2>(p, grid, st);
    case 7:
    case 8: return launch_ldg<T, 8, 1>(p, grid, st);
    default: {
      // the query as f32 (nv * QF = dim floats); oi_index_create refuses dim > OI_MAX_DIM, so this always fits
      static_assert(OI_MAX_DIM * sizeof(float) <= 96 * 1024, "OI_MAX_DIM must fit the wide-row kernel's query buffer");
      size_t smem = (size_t)p.nv * Elem<T>::QF * sizeof(float);
      if (smem > 96 * 1024) return cudaErrorInvalidValue;
      cudaError_t e = cudaFuncSetAttribute(cosine_scan_generic_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      if (e != cudaSuccess) return e;
      cosine_scan_generic_kernel<T><<<grid, kConsumerThreads, smem, st>>>(p);
      return cudaGetLastError();
    }
  }
}

// tile = a multiple of 32 rows (2 rows x 16 consumer warps) of at most 48 KB (16 rows for very wide rows); ring of <= 8 stages in 176 KB
static inline void bulk_tile_shape(uint32_t row_bytes, uint32_t *tile_rows, uint32_t *n_stages) {
  if (g_tile_rows_override > 0 && g_stages_override >= 2 &&
      (size_t)g_tile_rows_override * row_bytes * g_stages_override <= 176u * 1024u && g_tile_rows_override % 32 == 0) {
    *tile_rows = (uint32_t)g_tile_rows_override;
    *n_stages = (uint32_t)g_stages_override;
    return;
  }
  uint32_t tr = (49152u / row_bytes) & ~31u;
  if (tr < 16) tr = 16;
  if (tr > 256) tr = 256;
  uint32_t ns = (uint32_t)((176u * 1024u) / (tr * row_bytes));  // + 2 x 16.4 KB selection states <= 227 KB
  if (ns > 8) ns = 8;
  *tile_rows = tr;
  *n_stages = ns;
}

template <typename T, int NVL>
cudaError_t launch_bulk(const OiScanParams &p, uint32_t grid, cudaStream_t st) {
  const uint32_t row_bytes = p.nv * 16u;
  uint32_t tile_rows, n_stages;
  bulk_tile_shape(row_bytes, &tile_rows, &n_stages);
  if (n_stages < 2) return cudaErrorInvalidValue;
  const size_t smem = (size_t)n_stages * tile_rows * row_bytes + 2 * n_stages * sizeof(u64) + n_stages * sizeof(uint32_t);
  const bool exact = p.nv == 32u * NVL;
  cudaError_t e = exact ? cudaFuncSetAttribute(cosine_scan_bulk_kernel<T, NVL, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                        : cudaFuncSetAttribute(cosine_scan_bulk_kernel<T, NVL, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  if (exact) cosine_scan_bulk_kernel<T, NVL, true><<<grid, kBulkBlock, smem, st>>>(p, tile_rows, n_stages);
  else cosine_scan_bulk_kernel<T, NVL, false><<<grid, kBulkBlock, smem, st>>>(p, tile_rows, n_stages);
  return cudaGetLastError();
}

template <typename T>
cudaError_t dispatch_bulk(const OiScanParams &p, uint32_t grid, cudaStream_t st) {
  const uint32_t nvl = (p.nv + 31) / 32;
  switch (nvl) {
    case 1: return launch_bulk<T, 1>(p, grid, st);
    case 2: return launch_bulk<T, 2>(p, grid, st);
    case 3: return launch_bulk<T, 3>(p, grid, st);
    case 4: return launch_bulk<T, 4>(p, grid, st);
    case 5:
    case 6: return launch_bulk<T, 6>(p, grid, st);
    case 7:
    case 8: return launch_bulk<T, 8>(p, grid, st);
    default: return cudaErrorInvalidValue;
  }
}

// bulk-multi: the variant-1 tile shape with the ring cut down to leave room for kMultiQ selection states
static inline bool bulk_multi_shape(uint32_t row_bytes, uint32_t *tile_rows, uint32_t *n_stages, size_t *smem) {
  uint32_t tr = (49152u / row_bytes) & ~31u;
  if (tr < 32) return false;
  if (tr > 256) tr = 256;
  const size_t sel = (size_t)kMultiQ * sizeof(SelState);
  uint32_t ns = (uint32_t)((227u * 1024u - sel - 512u) / ((size_t)tr * row_bytes));
  if (ns > 8) ns = 8;
  if (ns < 2) return false;
  *tile_rows = tr;
  *n_stages = ns;
  *smem = (((size_t)ns * tr * row_bytes + ns * 20u + 15u) & ~(size_t)15) + sel;
  return true;
}

template <typename T, int NVL>
cudaError_t launch_bulk_multi_n(const OiScanParams &p, uint32_t grid, uint32_t tile_rows, uint32_t n_stages, size_t smem, cudaStream_t st) {
  cudaError_t e = cudaFuncSetAttribute(cosine_scan_bulk_multi_kernel<T, NVL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  cosine_scan_bulk_multi_kernel<T, NVL><<<grid, kBMBlock, smem, st>>>(p, tile_rows, n_stages);
  return cudaGetLastError();
}

template <typename T>
cudaError_t launch_bulk_multi(const OiScanParams &p, uint32_t grid, uint32_t tile_rows, uint32_t n_stages, size_t smem, cudaStream_t st) {
  switch ((p.nv + 31) / 32) {
    case 1: return launch_bulk_multi_n<T, 1>(p, grid, tile_rows, n_stages, smem, st);
    case 2: return launch_bulk_multi_n<T, 2>(p, grid, tile_rows, n_stages, smem, st);
    case 3: return launch_bulk_multi_n<T, 3>(p, grid, tile_rows, n_stages, smem, st);
    default: return cudaErrorInvalidValue;
  }
}

template <typename T>
cudaError_t launch_multi(const OiScanParams &p, uint32_t grid, cudaStream_t st) {
  const size_t smem = (size_t)kMultiQ * sizeof(SelState);
  const uint32_t nvl = (p.nv + 31) / 32;
  cudaError_t e;
  switch (nvl) {
    case 1:
      if ((e = cudaFuncSetAttribute(cosine_scan_multi_kernel<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
      cosine_scan_multi_kernel<T, 1><<<grid, kConsumerThreads, smem, st>>>(p);
      break;
    case 2:
      if ((e = cudaFuncSetAttribute(cosine_scan_multi_kernel<T, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
      cosine_scan_multi_kernel<T, 2><<<grid, kConsumerThreads, smem, st>>>(p);
      break;
    case 3:
      if ((e = cudaFuncSetAttribute(cosine_scan_multi_kernel<T, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
      cosine_scan_multi_kernel<T, 3><<<grid, kConsumerThreads, smem, st>>>(p);
      break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

__global__ void unpack_keys_kernel(const u64 *keys, uint32_t n, uint32_t *ids, float *scores) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  u64 key = keys[i];
  ids[i] = key ? oi_key_doc(key) : OI_NO_DOC_U32;
  scores[i] = key ? oi_key_score(key) : 0.0f;
}

// One CTA per query: exact top-k of `world` sorted lists (shards after the all-gather, or the per-item lists
// of the BM25 kernel), list r of query qi at gathered + (r * nq + qi) * k.
__global__ void __launch_bounds__(256) merge_shards_kernel(const u64 *gathered, uint32_t world, size_t rank_stride, uint32_t k, u64 *out,
                                                           const u64 *known) {
  __shared__ SelState S;
  const int tid = threadIdx.x;
  const uint32_t qi = blockIdx.x;
  merge_sorted_lists(S, gathered + (size_t)qi * k, world, rank_stride, k, tid, 256, 0, known ? __ldcg(known + qi) : 0ull);
  for (uint32_t i = tid; i < k; i += 256) out[(size_t)qi * k + i] = i < S.cnt ? S.buf[i] : 0ull;
}

}  // namespace

uint32_t oi_cosine_scan_max_grid(int num_sms) { return (uint32_t)num_sms * 2u; }

cudaError_t oi_launch_cosine_scan(const void *d_mat, uint32_t dtype, uint64_t n_rows, uint32_t dim,
                                  uint32_t doc_base, const float *d_queries, uint32_t nq, uint32_t k,
                                  const OiCosineWorkspace &ws, u64 *d_out_keys, int variant, int num_sms,
                                  cudaStream_t stream, uint64_t *launches, int multi_query) {
  const uint32_t esize = dtype == OI_DTYPE_F32 ? 4u : 2u;
  OiScanParams p;
  p.mat = reinterpret_cast<const uint4 *>(d_mat);
  p.n_rows = (uint32_t)n_rows;
  p.dim = dim;
  p.nv = dim * esize / 16u;
  p.doc_base = doc_base;
  p.k = k;
  if (multi_query && nq >= 2 && p.nv <= 96) {
    // groups of kMultiQ queries share one pass over the matrix
    uint32_t tile_rows = 0, n_stages = 0;
    size_t smem = 0;
    // the pipeline kernel has 96 registers per thread: the group's queries must fit in 48 of them
    const uint32_t q_regs = (uint32_t)kMultiQ * ((p.nv + 31) / 32) * (dtype == OI_DTYPE_F32 ? 4u : 8u);
    const bool bulk_multi = multi_query == 2 && q_regs <= 48 && bulk_multi_shape(p.nv * 16u, &tile_rows, &n_stages, &smem);
    uint32_t grid;
    if (bulk_multi) {  // cosine_scan_bulk_multi_kernel: one CTA per SM pulling tiles from a counter
      const uint32_t n_tiles = (uint32_t)((n_rows + tile_rows - 1) / tile_rows);
      grid = (uint32_t)num_sms;
      if (grid > n_tiles) grid = n_tiles ? n_tiles : 1;
      if (grid > ws.max_grid) grid = ws.max_grid;
      p.rows_per_cta = 0;
    } else {           // cosine_scan_multi_kernel: two CTAs per SM, contiguous row ranges
      grid = (uint32_t)num_sms * 2u;
      const uint32_t max_useful = (uint32_t)((n_rows + 63) / 64);
      if (grid > max_useful) grid = max_useful ? max_useful : 1;
      if (grid > ws.max_grid) grid = ws.max_grid;
      uint32_t rpc = (uint32_t)((n_rows + grid - 1) / grid);
      rpc = (rpc + 31u) & ~31u;
      if (rpc == 0) rpc = 32;  // an empty shard: one CTA that finds no rows
      p.rows_per_cta = rpc;
      grid = (uint32_t)((n_rows + rpc - 1) / rpc);
      if (grid == 0) grid = 1;
    }
    p.cand_stride = ws.max_grid * ws.k_stride;
    for (uint32_t g0 = 0; g0 < nq; g0 += kMultiQ) {
      p.nq = nq - g0 < (uint32_t)kMultiQ ? nq - g0 : (uint32_t)kMultiQ;
      p.q = d_queries + (size_t)g0 * dim;
      p.cand = ws.cand + (size_t)g0 * p.cand_stride;
      p.gthr = ws.gthr + g0;
      p.ticket = ws.ticket + g0;
      p.tile_ctr = ws.tile_ctr + g0;
      p.out_keys = d_out_keys + (size_t)g0 * k;
      cudaError_t e;
      if (bulk_multi) e = dtype == OI_DTYPE_F32 ? launch_bulk_multi<float>(p, grid, tile_rows, n_stages, smem, stream)
                                                : launch_bulk_multi<__nv_bfloat16>(p, grid, tile_rows, n_stages, smem, stream);
      else e = dtype == OI_DTYPE_F32 ? launch_multi<float>(p, grid, stream) : launch_multi<__nv_bfloat16>(p, grid, stream);
      if (e != cudaSuccess) return e;
      if (launches) ++*launches;
    }
    return cudaSuccess;
  }
  const bool bulk = variant == 1 && p.nv <= 256;
  uint32_t grid;
  if (bulk) {
    // one CTA per SM pulling tiles from a counter; never more CTAs than tiles
    uint32_t tile_rows, n_stages;
    bulk_tile_shape(p.nv * 16u, &tile_rows, &n_stages);
    const uint32_t n_tiles = (uint32_t)((n_rows + tile_rows - 1) / tile_rows);
    grid = (uint32_t)num_sms;
    if (grid > n_tiles) grid = n_tiles ? n_tiles : 1;
    if (grid > ws.max_grid) grid = ws.max_grid;
    p.rows_per_cta = 0;
  } else {
    // two CTAs per SM, each a contiguous row range, but never fewer than 64 rows per CTA
    grid = (uint32_t)num_sms * 2u;
    const uint32_t max_useful = (uint32_t)((n_rows + 63) / 64);
    if (grid > max_useful) grid = max_useful ? max_useful : 1;
    if (grid > ws.max_grid) grid = ws.max_grid;
    uint32_t rpc = (uint32_t)((n_rows + grid - 1) / grid);
    rpc = (rpc + 31u) & ~31u;
    if (rpc == 0) rpc = 32;  // an empty shard: one CTA that finds no rows
    p.rows_per_cta = rpc;
    grid = (uint32_t)((n_rows + rpc - 1) / rpc);
    if (grid == 0) grid = 1;
  }
  p.cand_stride = ws.max_grid * ws.k_stride;
  if (bulk) {
    // one persistent launch walks the whole batch: the epilogue (list merge) of query i overlaps
    // the streaming of query i+1
    p.nq = nq;
    p.q = d_queries;
    p.cand = ws.cand;
    p.gthr = ws.gthr;
    p.ticket = ws.ticket;
    p.tile_ctr = ws.tile_ctr;
    p.out_keys = d_out_keys;
    cudaError_t e = dtype == OI_DTYPE_F32 ? dispatch_bulk<float>(p, grid, stream) : dispatch_bulk<__nv_bfloat16>(p, grid, stream);
    if (e != cudaSuccess) return e;
    if (launches) ++*launches;
    return cudaSuccess;
  }
  p.nq = 1;
  for (uint32_t qi = 0; qi < nq; ++qi) {
    p.q = d_queries + (size_t)qi * dim;
    p.cand = ws.cand + (size_t)qi * p.cand_stride;
    p.gthr = ws.gthr + qi;
    p.ticket = ws.ticket + qi;
    p.tile_ctr = ws.tile_ctr + qi;
    p.out_keys = d_out_keys + (size_t)qi * k;
    cudaError_t e = dtype == OI_DTYPE_F32 ? dispatch_ldg<float>(p, grid, stream) : dispatch_ldg<__nv_bfloat16>(p, grid, stream);
    if (e != cudaSuccess) return e;
    if (launches) ++*launches;
  }
  return cudaSuccess;
}

cudaError_t oi_launch_unpack_keys(const u64 *d_keys, uint32_t n, uint32_t *d_ids, float *d_scores,
                                  cudaStream_t stream, uint64_t *launches) {
  if (n == 0) return cudaSuccess;
  unpack_keys_kernel<<<(n + 255) / 256, 256, 0, stream>>>(d_keys, n, d_ids, d_scores);
  if (launches) ++*launches;
  return cudaGetLastError();
}

cudaError_t oi_launch_merge_shards(const u64 *d_gathered, uint32_t world, uint32_t nq, uint32_t k,
                                   u64 *d_out, cudaStream_t stream, uint64_t *launches, size_t rank_stride, const u64 *d_known) {
  if (nq == 0) return cudaSuccess;
  merge_shards_kernel<<<nq, 256, 0, stream>>>(d_gathered, world, rank_stride ? rank_stride : (size_t)nq * k, k, d_out, d_known);
  if (launches) ++*launches;
  return cudaGetLastError();
}
