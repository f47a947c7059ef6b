// cosine_gemm.cu — batched cosine scoring on the 5th-generation tensor cores (BASELINE config 4:
// 10M x 768 bf16, 256 queries, top-100), with the top-k selection fused into the epilogue so that
// the nq x n_docs score matrix never exists in HBM.
//
//   S[q, d] = sum_j Q[q, j] * E[d, j]        Q: queries rounded to bf16 (SPEC §2), E: bf16 rows
//
// Mapping onto tcgen05.mma (kind::f16, cta_group::1, M = 128, N = 64, K = 16):
//   * A = 128 queries.  The whole query tile (128 x dim bf16) is written ONCE into tensor memory
//     (tcgen05.st, dim/2 of the 512 columns) and stays there: the A operand never touches shared
//     memory again, which leaves all of shared memory to the document stream.
//   * B = 64 document rows x 64 bf16 (one 128 B-swizzled TMA box, 8 KB) per pipeline stage, read
//     straight from the row-major embedding matrix by cp.async.bulk.tensor (UTMALDG).
//   * D = 128 x 64 f32 accumulators in tensor memory, double buffered (columns 384..511), so the
//     epilogue of document tile t overlaps the MMAs of tile t+1.
//   * a CTA owns one query tile and every n_ranges-th document tile; the n_qt CTAs that share a
//     document tile run side by side, so the second reader hits L2 and HBM is read once.
//   warp 0 = TMA producer, warp 1 = MMA issuer (one thread) + TMEM allocator, warps 2-5 = epilogue.
//
// Epilogue: thread r of the four epilogue warps owns TMEM lane r = query r of the tile.  It pulls
// the 64 scores of its query with tcgen05.ld, takes their maximum and compares it with the
// query's running threshold; only when the maximum passes does it look at individual scores and
// append (score, doc) keys to the (CTA, query) candidate list in global memory.  A list that
// could overflow is compacted to its best k by the warp (bitonic sort in shared memory) and the
// threshold raised.  A first short PROBE pass over a strided sample of the shard's tiles (~1 % of
// them) only records the maxima of groups of 8 scores; the k-th largest group maximum is a score
// at least k documents reach, i.e. a valid lower bound of every query's k-th best score, and seeds
// the one MAIN pass over all tiles.  The probe's merge also hands out a LADDER of tighter candidate
// bounds per query (its k/2-th, k/4-th, ... best group maximum).  During the main pass every score
// that passes the filter is counted, grid-wide, against the rungs above the current one
// (atomicAdd on 8 counters per query); as soon as k documents have reached a rung it is a valid
// bound too, and every CTA that polls the counter moves its filter up.  The filter so tightens
// geometrically while the pass runs -- about k survivors per rung, ~1000 keys per query in total --
// without any further launch.  (Round 1 used five passes of growing size, each with its own merge.)
//
//   algorithmic bytes per batch = n_docs * dim * 2        flops per batch = 2 * n_docs * dim * nq
#include <cuda.h>
#include <cuda_bf16.h>

#include <algorithm>

#include "handle.h"
#include "oi_common.cuh"
#include "oi_tcgen05.cuh"

struct OiGemm {
  __nv_bfloat16 *d_qb = nullptr;  // [n_qt_max * 128][dim] bf16 query tiles (zero padded)
  u64 *d_cand = nullptr;          // [max_lists][cap]
  uint32_t *d_cnt = nullptr;      // [max_lists]
  u64 *d_keys_a = nullptr;        // [max_batch][max_k] running result after a pass (ping)
  u64 *d_keys_b = nullptr;        // (pong)
  float *d_lvl_thr = nullptr;     // [max_batch][8] threshold ladder (ascending scores; -inf / +inf = no rung)
  uint32_t *d_lvl_cnt = nullptr;  // [max_batch][8] documents that reached a rung (main pass, grid-wide)
  uint32_t cap = 0;
  size_t max_lists = 0;
  CUtensorMap tmap;
  CUtensorMap tmap_pair;          // the same 3-D view with 32-row boxes (CTA pairs: each CTA loads half a tile)
  bool tma3d = false;
  bool pair_ok = false;
  bool ready = false;
};

namespace {

constexpr int kGemmThreads = 192;
constexpr uint32_t kTileDocs = 64;    // MMA N: documents per tile
constexpr uint32_t kKBlock = 64;      // bf16 elements per box row (128 B)
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kDCol0 = 384;      // two 64-column accumulators at 384 and 448
constexpr uint32_t kCapMax = 512;     // keys per (CTA, query) candidate list
constexpr uint32_t kMaxDim = 768;     // dim / 2 columns of TMEM hold the query tile
constexpr uint32_t kLevels = 8;       // rungs of the threshold ladder

struct GemmParams {
  const __nv_bfloat16 *qb;
  uint32_t n_rows, dim, doc_base, k, nq, n_qt, n_ranges;
  uint32_t tile_begin, tile_end;  // logical tiles [begin, end) covered by this launch; physical tile = logical * tile_mul
  uint32_t tile_mul;              // 1 for the main pass, the sampling stride for the probe pass
  uint32_t probe;                 // 1: record only the maxima of groups of 8 scores (score-only keys) for the threshold
  const float *lvl_thr;           // [nq][8] threshold ladder of the main pass (rung 0 = the probe's bound) or nullptr
  uint32_t *lvl_cnt;              // [nq][8] grid-wide counters of the documents that reached rungs 1..7
  u64 *cand;                      // [grid * 128][cap]
  uint32_t *cand_cnt;             // [grid * 128]
  uint32_t cap;
  float *dump;                    // tests: [nq][n_rows] raw scores, or nullptr
  uint32_t tma3d;                 // the tensor map is the 3-D (k-block-major) view: one TMA op per stage
  uint32_t debug;                 // timing experiments: bit 0 = no MMA issue, bit 1 = no TMA loads, bit 2 = no score filter (results are garbage),
                                  // bit 3 = the ladder stays on rung 0 (results stay exact)
};

__device__ __forceinline__ void warp_bitonic_desc(u64 *buf, uint32_t n, int lane) {
  for (uint32_t k = 2; k <= n; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t i = lane; i < (n >> 1); i += 32) {
        const uint32_t l = ((i & ~(j - 1)) << 1) | (i & (j - 1));
        const uint32_t r = l | j;
        const u64 a = buf[l], b = buf[r];
        const bool desc = (l & k) == 0;
        if ((a < b) == desc) { buf[l] = b; buf[r] = a; }
      }
      __syncwarp();
    }
  }
}

// The warp reduces list[0..n) to its best min(n, k) keys (sorted descending, written back to the
// front of the list).  Returns the k-th best key (0 when fewer than k are held).
__device__ __forceinline__ u64 warp_compact_list(u64 *list, uint32_t n, uint32_t k, u64 *scratch, int lane) {
  const uint32_t np2 = oi_next_pow2(n);
  for (uint32_t i = lane; i < np2; i += 32) scratch[i] = i < n ? __ldcg(list + i) : 0ull;
  __syncwarp();
  warp_bitonic_desc(scratch, np2, lane);
  const uint32_t keep = min(n, k);
  for (uint32_t i = lane; i < keep; i += 32) list[i] = scratch[i];
  const u64 thr = keep == k ? scratch[k - 1] : 0ull;
  __syncwarp();
  return thr;
}

// Slow path of the epilogue filter, OUT OF LINE on purpose: eight consecutive scores of one query (a group whose maximum
// passed the filter in some lane of the warp) are tested one by one and the survivors appended to the lane's candidate
// list; survivors that also reach the next rung of the threshold ladder are counted grid-wide.  Inlined and unrolled
// over the 64 scores of a tile this code was 15 KB per kernel: whenever survivors were frequent it evicted the MMA
// and TMA loops from the instruction cache (ncu: 9.5 "no instruction" stall cycles per issue, tensor pipe 13 % active)
// and a tile with a survivor cost the whole SM thousands of cycles.  Returns the new list length.
__device__ __noinline__ uint32_t gemm_open_group(uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, uint32_t s4, uint32_t s5,
                                                 uint32_t s6, uint32_t s7, u64 *buf, uint32_t cnt, float thr_s, u64 thr_key,
                                                 uint32_t doc, uint32_t doc_end, float nxt_s, const float *lvl, uint32_t *lvl_cnt,
                                                 uint32_t lv) {
  const uint32_t sv[8] = {s0, s1, s2, s3, s4, s5, s6, s7};
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const float sc = __uint_as_float(sv[e]);
    const u64 key = oi_make_key(sc, doc + e);
    const bool in_range = doc + e < doc_end;  // rows past the end of the shard are zero-filled by the TMA unit
    const bool ok = in_range && sc >= thr_s && key > thr_key;
    if (ok) buf[cnt] = key;
    cnt += ok ? 1u : 0u;
    if (in_range && sc >= nxt_s) {  // one more document on the rungs above (ascending: stop at the first it misses)
      for (uint32_t j = lv + 1; j < 8u; ++j) {
        if (!(sc >= __ldg(lvl + j))) break;
        atomicAdd(lvl_cnt + j, 1u);
      }
    }
  }
  return cnt;
}

// tests only (oi_debug_cosine_gemm_scores): eight raw scores of one query go to the dump matrix; out of line for the
// same code-size reason
__device__ __noinline__ void gemm_dump_group(uint32_t s0, uint32_t s1, uint32_t s2, uint32_t s3, uint32_t s4, uint32_t s5, uint32_t s6,
                                             uint32_t s7, float *dst, uint32_t n) {
  const uint32_t sv[8] = {s0, s1, s2, s3, s4, s5, s6, s7};
#pragma unroll
  for (int e = 0; e < 8; ++e)
    if ((uint32_t)e < n) dst[e] = __uint_as_float(sv[e]);
}

// Ring geometry for a row of NKB k-blocks (dim = 64 * NKB): the 192 KB ring holds 24 slabs of
// 64 rows x 128 B.  A stage = KBS slabs (one TMA op, one mbarrier); a tile = SPT stages; the ring
// holds TIF whole tiles, so inside a group of TIF tiles every stage index is a compile-time constant.
// RING = slabs in the ring: 24 (192 KB, the stand-alone kernel) or 12 (96 KB, the "lite" kernel that shares an SM
// with a BM25 CTA when the hybrid call overlaps its two legs).
// CG2 (CTA pairs): a slab holds this CTA's 32 of the tile's 64 rows (4 KB); the peer CTA holds the other 32.
template <int NKB, int RING, bool CG2 = false>
struct GemmShape {
  static_assert(RING % NKB == 0, "dim / 64 must divide the ring");
  static constexpr int KBS = (NKB % 4 == 0) ? 4 : (NKB % 2 == 0) ? 2 : 1;
  static constexpr int SPT = NKB / KBS;
  static constexpr int TIF = RING / NKB;
  static constexpr int STAGES = SPT * TIF;
  static constexpr uint32_t SLAB_BYTES = CG2 ? 4096u : 8192u;
  static constexpr uint32_t STAGE_BYTES = KBS * SLAB_BYTES;
  static constexpr uint32_t RING_BYTES = RING * SLAB_BYTES;
};
constexpr uint32_t kMaxStages = 24;
static_assert(true, "");

__device__ __forceinline__ uint32_t oi_elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xFFFFFFFF;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred;
}

// CG2: the kernel runs as clusters of two CTAs (the two SMs of a TPC).  CTA `rank` of a pair owns query tile
// 2 * (pair % (n_qt / 2)) + rank and HALF of every document tile (rows 32 * rank .. 32 * rank + 31); the leader (rank 0)
// issues ONE tcgen05.mma.cta_group::2 of M = 256 per k-step for both.  Every document row then enters exactly one SM
// (L2 -> SM traffic = the algorithmic bytes instead of twice that) and every SM reads half the B operand per flop from
// its shared memory (at M = 128, N = 64 the B reads plus the TMA writes used ~90 % of the shared-memory bandwidth and
// held the tensor pipe at 80 %: profiles/r02_ncu_cosine_gemm.md).
template <int NKB, int RING, bool EARLY, bool CG2 = false>
__device__ __forceinline__ void cosine_gemm_body(const CUtensorMap &tmap, const GemmParams &p) {
  using Sh = GemmShape<NKB, RING, CG2>;
  constexpr int KBS = Sh::KBS, SPT = Sh::SPT, TIF = Sh::TIF, STAGES = Sh::STAGES;
  extern __shared__ unsigned char s_raw[];
  unsigned char *sm = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(s_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char *s_stage = sm;                                                   // RING slabs x 8 KB, 1024 B aligned
  u64 *s_scratch = reinterpret_cast<u64 *>(sm + Sh::RING_BYTES);                 // 4 warps x cap keys
  u64 *s_full = s_scratch + 4 * kCapMax;
  u64 *s_empty = s_full + kMaxStages;
  u64 *s_tfull = s_empty + kMaxStages;  // [2] accumulator ready
  u64 *s_tempty = s_tfull + 2;          // [2] accumulator drained
  u64 *s_qready = s_tempty + 2;
  uint32_t *s_tmem = reinterpret_cast<uint32_t *>(s_qready + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // blockIdx.x = range * n_qt + qt in both layouts (a pair = two consecutive CTAs = two consecutive query tiles)
  const uint32_t qt = blockIdx.x % p.n_qt, range = blockIdx.x / p.n_qt;
  const uint32_t t0 = p.tile_begin + range;
  const uint32_t rank = CG2 ? oi_cluster_ctarank() : 0u;  // == qt & 1

  if (threadIdx.x == 0) {
    // CG2: full / tempty / qready are used in the LEADER only (both CTAs' copies report to it / arrive on it),
    // empty / tfull in each CTA (the leader's commits arrive on both)
    for (int s = 0; s < STAGES; ++s) { oi_mbar_init(&s_full[s], 1); oi_mbar_init(&s_empty[s], 1); }
    for (uint32_t b = 0; b < 2; ++b) { oi_mbar_init(&s_tfull[b], 1); oi_mbar_init(&s_tempty[b], CG2 ? 8 : 4); }
    oi_mbar_init(s_qready, CG2 ? 256 : 128);
    oi_mbar_fence_init();
  }
  if (warp == 1) { if (CG2) oi_tmem_alloc2(s_tmem, kTmemCols); else oi_tmem_alloc(s_tmem, kTmemCols); }
  oi_tc_fence_before();
  if (CG2) oi_cluster_sync(); else __syncthreads();  // the peer's barriers exist before anything is signalled to them
  oi_tc_fence_after();
  const uint32_t tmem = *s_tmem;

  // Warps 0 and 1 run their loops warp-uniformly and only the elected lane issues the TMA / MMA /
  // commit instructions: operands then live in uniform registers and one k-block costs a handful of
  // instructions (a single issuing thread must spend < 32 cycles per N = 64 MMA).
  if (warp == 0) {
    // ------------------------------- TMA producer ------------------------------------------------
    const bool leader = oi_elect_one();
    if (leader) oi_tma_prefetch_desc(&tmap);
    uint32_t grp = 0;
    for (uint32_t tb = t0; tb < p.tile_end; tb += TIF * p.n_ranges, ++grp) {
      const uint32_t ph = grp & 1u;
#pragma unroll
      for (int u = 0; u < TIF; ++u) {
        const uint32_t t = tb + u * p.n_ranges;
        if (t >= p.tile_end) break;
#pragma unroll
        for (int j = 0; j < SPT; ++j) {
          const int s = u * SPT + j;
          oi_mbar_wait(&s_empty[s], ph ^ 1u);
          if (leader) {
            if (CG2) {
              // each CTA brings its 32 rows of the tile; both report their bytes to the leader CTA's barrier, which
              // expects the two halves (a half that lands before the expectation is posted only makes the count
              // negative for a while: the phase cannot complete before the leader's own arrival)
              if (rank == 0) oi_mbar_expect_tx(&s_full[s], 2u * Sh::STAGE_BYTES);
              oi_tma_load_3d_pair(s_stage + (size_t)s * Sh::STAGE_BYTES, &tmap, 0, (int32_t)(t * p.tile_mul * kTileDocs + rank * 32u), j * KBS,
                                  &s_full[s]);
            } else if (p.debug & 2u) {
              oi_mbar_arrive(&s_full[s]);
            } else {
              oi_mbar_expect_tx(&s_full[s], Sh::STAGE_BYTES);
              // rows past the end of the shard are zero-filled by the TMA unit
              if (p.tma3d) {
                oi_tma_load_3d(s_stage + (size_t)s * Sh::STAGE_BYTES, &tmap, 0, (int32_t)(t * p.tile_mul * kTileDocs), j * KBS, &s_full[s]);
              } else {
#pragma unroll
                for (int kk = 0; kk < KBS; ++kk)
                  oi_tma_load_2d(s_stage + (size_t)s * Sh::STAGE_BYTES + kk * 8192, &tmap, (j * KBS + kk) * (int)kKBlock,
                                 (int32_t)(t * p.tile_mul * kTileDocs), &s_full[s]);
              }
            }
          }
        }
      }
    }
  } else if (warp == 1 && (!CG2 || rank == 0)) {
    // ------------------------------- MMA issuer (CG2: in the leader CTA only) ----------------------
    const bool leader = oi_elect_one();
    constexpr uint32_t idesc = oi_umma_idesc_bf16(CG2 ? 256 : 128, kTileDocs);
    constexpr uint32_t kSlab16 = Sh::SLAB_BYTES / 16;  // descriptor address units per slab
    const uint64_t desc0 = oi_umma_smem_desc_sw128(oi_smem_u32(s_stage));
    if (CG2) oi_mbar_wait_cluster(s_qready, 0); else oi_mbar_wait(s_qready, 0);
    oi_tc_fence_after();
    uint32_t grp = 0, tl = 0;
    for (uint32_t tb = t0; tb < p.tile_end; tb += TIF * p.n_ranges, ++grp) {
      const uint32_t ph = grp & 1u;
#pragma unroll
      for (int u = 0; u < TIF; ++u) {
        const uint32_t t = tb + u * p.n_ranges;
        if (t >= p.tile_end) break;
        const uint32_t b = tl & 1u, bph = (tl >> 1) & 1u;
        ++tl;
        if (CG2) oi_mbar_wait_cluster(&s_tempty[b], bph ^ 1u); else oi_mbar_wait(&s_tempty[b], bph ^ 1u);
        oi_tc_fence_after();
        const uint32_t d_addr = tmem + kDCol0 + b * kTileDocs;
#pragma unroll
        for (int j = 0; j < SPT; ++j) {
          const int s = u * SPT + j;
          oi_mbar_wait(&s_full[s], ph);
          oi_tc_fence_after();
          if (leader) {
            if (!CG2 && (p.debug & 1u)) {
              oi_mbar_arrive(&s_empty[s]);
              if (j == SPT - 1) oi_mbar_arrive(&s_tfull[b]);
            } else {
#pragma unroll
              for (int kk = 0; kk < KBS; ++kk) {
#pragma unroll
                for (int ks = 0; ks < 4; ++ks) {
                  // A: 16 bf16 of K = 8 TMEM columns; B: slab (s * KBS + kk), 32 B per k-step inside the swizzle atom
                  const int kbi = j * KBS + kk;
                  const uint64_t db = desc0 + (uint64_t)((s * KBS + kk) * kSlab16 + ks * 2);
                  if (CG2) oi_umma2_ts_bf16(d_addr, tmem + (uint32_t)((kbi * 4 + ks) * 8), db, idesc, (kbi | ks) != 0 ? 1u : 0u);
                  else oi_umma_ts_bf16(d_addr, tmem + (uint32_t)((kbi * 4 + ks) * 8), db, idesc, (kbi | ks) != 0 ? 1u : 0u);
                }
              }
              // the stage is free (in both CTAs) once these MMAs have read it; the accumulator is ready in both
              if (CG2) oi_umma2_commit_mc(&s_empty[s], 3u); else oi_umma_commit(&s_empty[s]);
              if (j == SPT - 1) { if (CG2) oi_umma2_commit_mc(&s_tfull[b], 3u); else oi_umma_commit(&s_tfull[b]); }
            }
          }
        }
      }
    }
  } else if (warp >= 2) {
    // ------------------------------- epilogue: one thread per query -------------------------------
    const uint32_t quarter = (uint32_t)warp & 3u;  // TMEM lanes this warp may touch: 32 * (warp % 4)
    const uint32_t row = quarter * 32 + lane;
    const uint32_t lane_taddr = tmem + ((quarter * 32u) << 16);
    {
      // the prep kernel stored the tile as [quarter][32-column chunk][lane][32 x u32]: one chunk of one
      // warp is 4 KB contiguous, 128 B per lane
      const uint32_t n_chunks = p.dim / 64;
      const uint4 *qsrc = reinterpret_cast<const uint4 *>(p.qb) + ((size_t)(qt * 4 + quarter) * n_chunks * 32 + lane) * 8;
#pragma unroll 1
      for (uint32_t ch = 0; ch < n_chunks; ++ch) {  // once per launch: no prefetch, no unrolling (code size)
        uint32_t r[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const uint4 x = __ldg(qsrc + (size_t)ch * 256 + j);
          r[4 * j] = x.x; r[4 * j + 1] = x.y; r[4 * j + 2] = x.z; r[4 * j + 3] = x.w;
        }
        oi_tmem_st32(lane_taddr + ch * 32, r);
      }
      oi_tmem_wait_st();
      oi_tc_fence_before();
      if (CG2) oi_mbar_arrive_cluster(s_qready, 0u); else oi_mbar_arrive(s_qready);
    }
    const uint32_t q = qt * 128 + row;
    const bool qv = q < p.nq;
    const uint32_t cap = p.cap;
    const size_t list = (size_t)blockIdx.x * 128 + row;
    u64 *buf = p.cand + list * cap;
    u64 *scratch = s_scratch + (size_t)(warp - 2) * kCapMax;
    uint32_t cnt = 0;
    // threshold ladder: rung 0 is valid from the start, rung lv + 1 once its grid-wide counter reaches k
    const bool ladder = qv && p.lvl_thr != nullptr && !p.probe;
    const float *my_lvl = p.lvl_thr + (size_t)(qv ? q : 0) * kLevels;
    uint32_t *my_cnt = p.lvl_cnt + (size_t)(qv ? q : 0) * kLevels;
    uint32_t lv = 0;
    const bool climb = ladder && !(p.debug & 8u);
    float thr_s = ladder ? __ldg(my_lvl) : (qv ? -INFINITY : INFINITY);  // lanes without a query never pass the filter
    float nxt_s = ladder ? __ldg(my_lvl + 1) : INFINITY;  // the rung being counted
    u64 thr_key = (ladder && thr_s > -INFINITY) ? ((u64)oi_ord(thr_s) << 32) : 0ull;

    uint32_t tl = 0;
    for (uint32_t t = t0; t < p.tile_end; t += p.n_ranges, ++tl) {
      const uint32_t b = tl & 1u, bph = (tl >> 1) & 1u;
      // every 4th tile: has the next rung been reached by k documents?  (requested now, consumed after the tile)
      const bool poll = climb && (tl & 3u) == 3u && lv + 1 < kLevels;
      uint32_t polled = 0;
      if (poll) asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(polled) : "l"(my_cnt + lv + 1) : "memory");
      oi_mbar_wait(&s_tfull[b], bph);
      oi_tc_fence_after();
      const uint32_t doc0 = t * p.tile_mul * kTileDocs;
      const uint32_t n_valid = min(kTileDocs, p.n_rows - doc0);
      // NH = 1 (stand-alone kernel): all 64 scores of the tile are pulled at once and the accumulator is released as
      // soon as they are in registers -- the MMAs of tile t + 2 never wait for this warp's arithmetic (holding the
      // accumulator through two TMEM round trips and the filter cost ~6 %: profiles/r02_gemm_ab.md).
      // NH = 2 (lite kernel, 128 registers): two halves of 32 columns, released after the second.
      constexpr int NH = EARLY ? 1 : 2, W = 64 / NH;
#pragma unroll
      for (int hf = 0; hf < NH; ++hf) {
        uint32_t v[W];
        oi_tmem_ld32(lane_taddr + kDCol0 + b * kTileDocs + hf * W, v);
        if (EARLY) oi_tmem_ld32(lane_taddr + kDCol0 + b * kTileDocs + 32, v + (EARLY ? 32 : 0));
        oi_tmem_wait_ld();
        if (EARLY || hf == NH - 1) {
          oi_tc_fence_before();
          __syncwarp();
          // the scores are in registers: the accumulator may be overwritten (CG2: the leader's issuer waits for both CTAs)
          if (lane == 0) { if (CG2) oi_mbar_arrive_cluster(&s_tempty[b], 0u); else oi_mbar_arrive(&s_tempty[b]); }
        }
        if (p.dump) {  // warp-uniform
#pragma unroll
          for (int g = 0; g < W / 8; ++g) {
            const uint32_t c0 = (uint32_t)(hf * W + 8 * g);
            gemm_dump_group(v[8 * g], v[8 * g + 1], v[8 * g + 2], v[8 * g + 3], v[8 * g + 4], v[8 * g + 5], v[8 * g + 6], v[8 * g + 7],
                            p.dump + (size_t)(qv ? q : 0) * p.n_rows + doc0 + c0, (qv && n_valid > c0) ? n_valid - c0 : 0u);
          }
        }
        // two-level filter: maxima of groups of 8 scores, then their maximum.  Most tiles stop at the single compare.
        // Every branch below is WARP-UNIFORM (ballots) and the per-score work inside an opened group is predicated: the
        // first version branched per lane and per score, 64 divergent regions per tile, and a tile with a survivor cost
        // the warp more than a thousand cycles (profiles/r02_gemm_ab.md).  Lanes without a query carry thr_s = +inf.
        constexpr int NG = W / 8;
        float gm[NG];
#pragma unroll
        for (int g = 0; g < NG; ++g) {
          const float a = fmaxf(fmaxf(__uint_as_float(v[8 * g]), __uint_as_float(v[8 * g + 1])), __uint_as_float(v[8 * g + 2]));
          const float c = fmaxf(fmaxf(__uint_as_float(v[8 * g + 3]), __uint_as_float(v[8 * g + 4])), __uint_as_float(v[8 * g + 5]));
          gm[g] = fmaxf(fmaxf(a, c), fmaxf(__uint_as_float(v[8 * g + 6]), __uint_as_float(v[8 * g + 7])));
        }
        if (p.probe) {
          // probe pass: a group maximum is the score of one real document and the groups are disjoint, so the k-th
          // largest of them is a score at least k documents reach.  Score-only keys (doc field 0).
#pragma unroll
          for (int g = 0; g < NG; ++g) {
            // a partial last tile is left out of the sample: its zero-filled columns are not documents
            const bool ok = qv && n_valid == kTileDocs;
            if (ok) buf[cnt] = (u64)oi_ord(gm[g]) << 32;
            cnt += ok ? 1u : 0u;
          }
        } else if (!(p.debug & 4u)) {
          float m = gm[0];
#pragma unroll
          for (int g = 1; g < NG; ++g) m = fmaxf(m, gm[g]);
          if (__any_sync(0xFFFFFFFFu, m >= thr_s)) {
            const float cnt_s = climb ? nxt_s : INFINITY;
#pragma unroll
            for (int g = 0; g < NG; ++g) {
              if (__any_sync(0xFFFFFFFFu, gm[g] >= thr_s))
                cnt = gemm_open_group(v[8 * g], v[8 * g + 1], v[8 * g + 2], v[8 * g + 3], v[8 * g + 4], v[8 * g + 5], v[8 * g + 6],
                                      v[8 * g + 7], buf, cnt, thr_s, thr_key, p.doc_base + doc0 + hf * W + 8 * g, p.doc_base + p.n_rows,
                                      cnt_s, my_lvl, my_cnt, lv);
            }
          }
        }
      }
      if (poll && polled >= p.k) {  // k documents reached the next rung: it bounds the k-th best score from below
        ++lv;
        const u64 cand_key = (u64)oi_ord(nxt_s) << 32;
        if (cand_key > thr_key) { thr_key = cand_key; thr_s = nxt_s; }
        nxt_s = lv + 1 < kLevels ? __ldg(my_lvl + lv + 1) : INFINITY;
      }

      // a list that could overflow during the next tile is reduced to its best k by the whole warp
      uint32_t mask = __ballot_sync(0xFFFFFFFFu, cnt + kTileDocs > cap);
      while (mask) {
        const int l = __ffs(mask) - 1;
        mask &= mask - 1;
        const uint32_t n_l = __shfl_sync(0xFFFFFFFFu, cnt, l);
        u64 *list_l = p.cand + ((size_t)blockIdx.x * 128 + quarter * 32 + l) * cap;
        __syncwarp();
        const u64 thr_l = warp_compact_list(list_l, n_l, p.k, scratch, lane);
        if (lane == l) {
          cnt = min(n_l, p.k);
          if (thr_l > thr_key) { thr_key = thr_l; thr_s = oi_key_score(thr_l); }
        }
      }
    }
    p.cand_cnt[list] = qv ? cnt : 0u;
  }

  oi_tc_fence_before();
  if (CG2) oi_cluster_sync(); else __syncthreads();  // CG2: no CTA leaves while its peer may still signal its barriers
  if (warp == 1) {
    oi_tc_fence_after();
    if (CG2) oi_tmem_dealloc2(tmem, kTmemCols); else oi_tmem_dealloc(tmem, kTmemCols);
  }
}

// Two entry points over the same body.  The stand-alone kernel owns its SM (192 KB ring, any register count).  The
// "lite" kernel (96 KB ring) is capped at 128 registers per thread so that 192 x 128 = 24.5 k registers and 116 KB of
// shared memory leave room on the SM for one BM25 CTA (hybrid overlap, api.cu).
template <int NKB, int RING>
__global__ void __launch_bounds__(kGemmThreads, 1)
    cosine_gemm_kernel(const __grid_constant__ CUtensorMap tmap, const GemmParams p) {
  cosine_gemm_body<NKB, RING, true>(tmap, p);
}
template <int NKB, int RING>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kGemmThreads, 1)
    cosine_gemm_pair_kernel(const __grid_constant__ CUtensorMap tmap, const GemmParams p) {
  cosine_gemm_body<NKB, RING, true, true>(tmap, p);
}
template <int NKB, int RING>
__global__ void __maxnreg__(128)
    cosine_gemm_lite_kernel(const __grid_constant__ CUtensorMap tmap, const GemmParams p) {
  cosine_gemm_body<NKB, RING, false>(tmap, p);
}

// f32 queries -> bf16 pairs (RNE, SPEC §2), zero rows up to a multiple of 128, stored in the order the
// epilogue warps feed tcgen05.st: [query tile][lane quarter][32-column chunk][lane][32 x u32], where 32-bit
// column c of a row holds elements (2c, 2c + 1) with 2c in the low half.
__global__ void gemm_prep_queries_kernel(const float *q, uint32_t nq, uint32_t rows, uint32_t dim, uint32_t *qb) {
  const uint32_t n_chunks = dim / 64;
  const size_t n = (size_t)rows * dim / 2;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t w = (uint32_t)(i & 31), lane = (uint32_t)((i >> 5) & 31);
    const size_t rest = i >> 10;
    const uint32_t chunk = (uint32_t)(rest % n_chunks);
    const size_t tq = rest / n_chunks;  // tile * 4 + quarter
    const size_t row = tq * 32 + lane;
    const uint32_t c = chunk * 32 + w;
    uint32_t packed = 0;
    if (row < nq) {
      const float2 f = *reinterpret_cast<const float2 *>(q + row * dim + 2 * c);
      const __nv_bfloat16 lo = __float2bfloat16_rn(f.x), hi = __float2bfloat16_rn(f.y);
      packed = (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
    }
    qb[i] = packed;
  }
}

struct MergeState {
  u64 buf[OI_SEL_CAP];
  u64 thr;
  uint32_t cnt;
};

// One CTA per query: exact top-k over the query's n_ranges candidate lists (+ the sorted list of the
// earlier passes).  out[q][k] sorted descending; lvl_thr / lvl_cnt (probe merge only): see the end.  The lists are walked as
// one flat key sequence (prefix sums of the list lengths in shared memory), a buffer-load at a time,
// every thread holding up to 8 independent loads in flight.
constexpr uint32_t kMergeMaxLists = 1020;
__global__ void __launch_bounds__(256) gemm_merge_kernel(const u64 *cand, const uint32_t *cnts, uint32_t cap, uint32_t n_ranges,
                                                         uint32_t n_qt, uint32_t k, const u64 *prev, u64 *out, float *lvl_thr,
                                                         uint32_t *lvl_cnt) {
  __shared__ MergeState S;
  __shared__ uint32_t s_pre[kMergeMaxLists + 4];
  __shared__ uint32_t s_wsum[8];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t q = blockIdx.x, qt = q / 128, rl = q % 128;
  // exclusive prefix sums of the list lengths: thread t owns lists 4t .. 4t+3
  uint32_t c[4], tsum = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const uint32_t r = tid * 4 + u;
    c[u] = r < n_ranges ? min(cnts[((size_t)r * n_qt + qt) * 128 + rl], cap) : 0u;
    tsum += c[u];
  }
  uint32_t x = tsum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
    if (lane >= o) x += y;
  }
  if (lane == 31) s_wsum[warp] = x;
  // the earlier passes' list is already the best k of its documents: it seeds the buffer
  uint32_t seed = 0;
  if (prev) {
    for (uint32_t i = tid; i < k; i += 256) S.buf[i] = prev[(size_t)q * k + i];
    seed = k;
  }
  if (tid == 0) { S.cnt = seed; S.thr = 0ull; }
  __syncthreads();
  uint32_t excl = x - tsum;
  for (int w = 0; w < warp; ++w) excl += s_wsum[w];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const uint32_t r = tid * 4 + u;
    if (r <= n_ranges) s_pre[r] = excl;
    excl += c[u];
  }
  __syncthreads();
  if (prev) oi_sel_compact(S.buf, &S.cnt, &S.thr, k, tid, 256, 0);  // sets thr when k real keys are held
  const uint32_t total = s_pre[n_ranges];
  uint32_t f0 = 0;
  while (f0 < total) {
    const uint32_t len = min(total - f0, (uint32_t)OI_SEL_CAP - S.cnt);
    const u64 thr = S.thr;
    __syncthreads();  // (cnt, thr) snapshot taken by everybody before anybody pushes
    u64 keys[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const uint32_t f = f0 + tid + u * 256;
      keys[u] = 0ull;
      if (f < f0 + len) {
        uint32_t lo = 0, hi = n_ranges;  // s_pre[lo] <= f < s_pre[hi]
        while (hi - lo > 1) {
          const uint32_t mid = (lo + hi) >> 1;
          if (s_pre[mid] <= f) lo = mid; else hi = mid;
        }
        keys[u] = __ldcg(cand + (((size_t)lo * n_qt + qt) * 128 + rl) * cap + (f - s_pre[lo]));
      }
    }
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const bool pass = keys[u] > thr;
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, pass);
      if (m) {
        uint32_t base = 0;
        if (lane == 0) base = atomicAdd(&S.cnt, (uint32_t)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, 0);
        if (pass) S.buf[base + __popc(m & ((1u << lane) - 1))] = keys[u];
      }
    }
    f0 += len;
    __syncthreads();
    if (S.cnt > OI_SEL_CAP / 2 || f0 >= total) oi_sel_compact(S.buf, &S.cnt, &S.thr, k, tid, 256, 0);
  }
  for (uint32_t i = tid; i < k; i += 256) out[(size_t)q * k + i] = i < S.cnt ? S.buf[i] : 0ull;
  // probe merge: the ladder of the main pass.  Rung j = the (k >> j)-th best group maximum: a score (k >> j) / (sample
  // fraction) documents are expected to reach, valid as a bound once k documents HAVE reached it (counted in the main
  // pass).  Rung 0 (the k-th best) is valid at once.  Fewer than k group maxima: no bound at all.
  if (lvl_thr && tid < (int)kLevels) {
    const uint32_t r = k >> tid;
    float t = tid == 0 ? -INFINITY : INFINITY;
    if (S.cnt == k && r >= 1) t = oi_key_score(S.buf[r - 1]);
    lvl_thr[(size_t)q * kLevels + tid] = t;
    lvl_cnt[(size_t)q * kLevels + tid] = 0u;
  }
}

size_t gemm_smem_bytes(int ring, bool pair = false) {
  return 1024 + (size_t)ring * (pair ? 4096 : 8192) + 4 * kCapMax * sizeof(u64) + (2 * kMaxStages + 5) * sizeof(u64) + 16;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

}  // namespace

void oi_gemm_free(oi_index *h) {
  OiGemm *g = h->gemm;
  if (!g) return;
  cudaFree(g->d_qb); cudaFree(g->d_cand); cudaFree(g->d_cnt); cudaFree(g->d_keys_a); cudaFree(g->d_keys_b); cudaFree(g->d_lvl_thr); cudaFree(g->d_lvl_cnt);
  delete g;
  h->gemm = nullptr;
}

bool oi_gemm_eligible(const oi_index *h, uint32_t nq, uint32_t k) {
  const uint32_t cap = h->gemm_cap ? (uint32_t)h->gemm_cap : kCapMax;
  return h->desc.dtype == OI_DTYPE_BF16 && h->desc.dim % kKBlock == 0 && h->desc.dim <= kMaxDim &&
         24 % (h->desc.dim / kKBlock) == 0 && h->desc.n_docs > 0 &&
         h->desc.n_docs < 0x7FFFFFC0ull && k + kTileDocs <= cap && nq >= 1;
}

// lazily: workspace + the tensor map of the embedding matrix
static oi_status gemm_prepare(oi_index *h) {
  if (h->gemm && h->gemm->ready) return OI_OK;
  if (!h->gemm) h->gemm = new OiGemm();
  OiGemm *g = h->gemm;
  const size_t B = h->desc.max_batch, K = h->desc.max_k, dim = h->desc.dim;
  const size_t n_qt_max = (B + 127) / 128;
  g->cap = kCapMax;
  g->max_lists = (size_t)std::max<size_t>((size_t)h->num_sms, n_qt_max) * 128;
  OI_CK(cudaMalloc(&g->d_qb, n_qt_max * 128 * dim * sizeof(__nv_bfloat16)));
  OI_CK(cudaMalloc(&g->d_cand, g->max_lists * g->cap * sizeof(u64)));
  OI_CK(cudaMalloc(&g->d_cnt, g->max_lists * sizeof(uint32_t)));
  OI_CK(cudaMalloc(&g->d_keys_a, B * K * sizeof(u64)));
  OI_CK(cudaMalloc(&g->d_keys_b, B * K * sizeof(u64)));
  OI_CK(cudaMalloc(&g->d_lvl_thr, B * kLevels * sizeof(float)));
  OI_CK(cudaMalloc(&g->d_lvl_cnt, B * kLevels * sizeof(uint32_t)));

  void *fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  OI_CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (!fn || qres != cudaDriverEntryPointSuccess) return h->fail(OI_ERR_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
  // 3-D view (64 elements, rows, k-blocks): one TMA op brings KBS consecutive 128 B column slabs of 64 rows,
  // each landing as its own swizzled 8 KB slab.  If the driver rejects the view, fall back to one 2-D box per slab.
  const uint32_t nkb = (uint32_t)(dim / kKBlock);
  const uint32_t kbs = nkb % 4 == 0 ? 4 : nkb % 2 == 0 ? 2 : 1;
  const cuuint32_t estr[3] = {1, 1, 1};
  {
    const cuuint64_t gdim[3] = {kKBlock, (cuuint64_t)h->desc.n_docs, nkb};
    const cuuint64_t gstride[2] = {(cuuint64_t)dim * sizeof(__nv_bfloat16), kKBlock * sizeof(__nv_bfloat16)};
    const cuuint32_t box[3] = {kKBlock, kTileDocs, kbs};
    CUresult cr = ((EncodeTiledFn)fn)(&g->tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, h->d_emb, gdim, gstride, box, estr,
                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    g->tma3d = cr == CUDA_SUCCESS;
    if (g->tma3d) {
      const cuuint32_t box2[3] = {kKBlock, kTileDocs / 2, kbs};
      cr = ((EncodeTiledFn)fn)(&g->tmap_pair, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, h->d_emb, gdim, gstride, box2, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
      g->pair_ok = cr == CUDA_SUCCESS;
    }
  }
  if (!g->tma3d || h->gemm_force_2d) {
    const cuuint64_t gdim[2] = {(cuuint64_t)dim, (cuuint64_t)h->desc.n_docs};
    const cuuint64_t gstride[1] = {(cuuint64_t)dim * sizeof(__nv_bfloat16)};
    const cuuint32_t box[2] = {kKBlock, kTileDocs};
    CUresult cr = ((EncodeTiledFn)fn)(&g->tmap, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, h->d_emb, gdim, gstride, box, estr,
                                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) return h->fail(OI_ERR_CUDA, "cuTensorMapEncodeTiled failed (CUresult %d)", (int)cr);
    g->tma3d = false;
  }
  const int smem = (int)gemm_smem_bytes(24), smem_lite = (int)gemm_smem_bytes(12);
#define OI_GEMM_ATTR(KERNEL, NKB, RING, BYTES) OI_CK(cudaFuncSetAttribute(KERNEL<NKB, RING>, cudaFuncAttributeMaxDynamicSharedMemorySize, BYTES))
  OI_GEMM_ATTR(cosine_gemm_kernel, 1, 24, smem); OI_GEMM_ATTR(cosine_gemm_kernel, 2, 24, smem); OI_GEMM_ATTR(cosine_gemm_kernel, 3, 24, smem);
  OI_GEMM_ATTR(cosine_gemm_kernel, 4, 24, smem); OI_GEMM_ATTR(cosine_gemm_kernel, 6, 24, smem); OI_GEMM_ATTR(cosine_gemm_kernel, 8, 24, smem);
  OI_GEMM_ATTR(cosine_gemm_kernel, 12, 24, smem);
  OI_GEMM_ATTR(cosine_gemm_lite_kernel, 1, 12, smem_lite); OI_GEMM_ATTR(cosine_gemm_lite_kernel, 2, 12, smem_lite);
  OI_GEMM_ATTR(cosine_gemm_lite_kernel, 3, 12, smem_lite); OI_GEMM_ATTR(cosine_gemm_lite_kernel, 4, 12, smem_lite);
  OI_GEMM_ATTR(cosine_gemm_lite_kernel, 6, 12, smem_lite); OI_GEMM_ATTR(cosine_gemm_lite_kernel, 12, 12, smem_lite);
  {
    const int smem_p24 = (int)gemm_smem_bytes(24, true), smem_p48 = (int)gemm_smem_bytes(48, true);
    OI_GEMM_ATTR(cosine_gemm_pair_kernel, 1, 24, smem_p24); OI_GEMM_ATTR(cosine_gemm_pair_kernel, 2, 24, smem_p24);
    OI_GEMM_ATTR(cosine_gemm_pair_kernel, 3, 24, smem_p24); OI_GEMM_ATTR(cosine_gemm_pair_kernel, 4, 24, smem_p24);
    OI_GEMM_ATTR(cosine_gemm_pair_kernel, 6, 24, smem_p24); OI_GEMM_ATTR(cosine_gemm_pair_kernel, 8, 24, smem_p24);
    OI_GEMM_ATTR(cosine_gemm_pair_kernel, 12, 24, smem_p24); OI_GEMM_ATTR(cosine_gemm_pair_kernel, 12, 48, smem_p48);
  }
#undef OI_GEMM_ATTR
  g->ready = true;
  return OI_OK;
}

// the "lite" kernel (96 KB ring) exists for the row widths whose tile fits it
bool oi_gemm_lite_ok(const oi_index *h) { return 12 % (h->desc.dim / kKBlock) == 0; }

static oi_status gemm_launch(oi_index *h, uint32_t nq, uint32_t n_qt, uint32_t n_ranges, uint32_t k, uint32_t cap,
                             uint32_t tile_begin, uint32_t tile_end, uint32_t tile_mul, bool probe, const float *lvl_thr, float *dump,
                             bool lite, bool pair, cudaStream_t st) {
  OiGemm *g = h->gemm;
  GemmParams p;
  p.qb = g->d_qb;
  p.n_rows = (uint32_t)h->desc.n_docs; p.dim = h->desc.dim; p.doc_base = (uint32_t)h->desc.doc_base;
  p.k = k; p.nq = nq; p.n_qt = n_qt; p.n_ranges = n_ranges;
  p.tile_begin = tile_begin; p.tile_end = tile_end; p.tile_mul = tile_mul; p.probe = probe ? 1u : 0u;
  p.lvl_thr = lvl_thr; p.lvl_cnt = g->d_lvl_cnt; p.cand = g->d_cand; p.cand_cnt = g->d_cnt; p.cap = cap; p.dump = dump;
  p.debug = (uint32_t)h->gemm_debug;
  p.tma3d = g->tma3d ? 1u : 0u;
  const uint32_t grid = n_ranges * n_qt;
  const uint32_t nkb = h->desc.dim / kKBlock;
  if (lite && 12 % nkb != 0) lite = false;
  if (pair) {  // CTA pairs: clusters of two, tcgen05.mma.cta_group::2
    p.tma3d = 1u;
    const bool deep = nkb == 12 && h->gemm_pair_ring == 48;
    const size_t smem_p = gemm_smem_bytes(deep ? 48 : 24, true);
#define OI_GEMM_PAIR(NKB) case NKB: cosine_gemm_pair_kernel<NKB, 24><<<grid, kGemmThreads, smem_p, st>>>(g->tmap_pair, p); break;
    if (deep) {
      cosine_gemm_pair_kernel<12, 48><<<grid, kGemmThreads, smem_p, st>>>(g->tmap_pair, p);
    } else {
      switch (nkb) {
        OI_GEMM_PAIR(1) OI_GEMM_PAIR(2) OI_GEMM_PAIR(3) OI_GEMM_PAIR(4) OI_GEMM_PAIR(6) OI_GEMM_PAIR(8) OI_GEMM_PAIR(12)
        default: return h->fail(OI_ERR_UNSUPPORTED, "internal: dim %u has no tensor-core kernel", h->desc.dim);
      }
    }
#undef OI_GEMM_PAIR
    ++h->launches;
    OI_CK(cudaGetLastError());
    return OI_OK;
  }
  const size_t smem = gemm_smem_bytes(lite ? 12 : 24);
#define OI_GEMM_GO(NKB)                                                                       \
  case NKB:                                                                                   \
    if (lite) cosine_gemm_lite_kernel<(12 % NKB == 0 ? NKB : 12), 12><<<grid, kGemmThreads, smem, st>>>(g->tmap, p); \
    else cosine_gemm_kernel<NKB, 24><<<grid, kGemmThreads, smem, st>>>(g->tmap, p);           \
    break;
  switch (nkb) {
    OI_GEMM_GO(1) OI_GEMM_GO(2) OI_GEMM_GO(3) OI_GEMM_GO(4) OI_GEMM_GO(6) OI_GEMM_GO(8) OI_GEMM_GO(12)
    default: return h->fail(OI_ERR_UNSUPPORTED, "internal: dim %u has no tensor-core kernel", h->desc.dim);
  }
#undef OI_GEMM_GO
  ++h->launches;
  OI_CK(cudaGetLastError());
  return OI_OK;
}

// Shard-local top-k lists d_out_keys[nq][k] (sorted, global doc ids) of nq f32 queries on the device.
oi_status oi_gemm_local_keys(oi_index *h, const float *d_queries, uint32_t nq, uint32_t k, u64 *d_out_keys, float *d_dump,
                             cudaStream_t st, bool lite, uint32_t max_ctas) {
  oi_status s = gemm_prepare(h);
  if (s) return s;
  OiGemm *g = h->gemm;
  const uint32_t n_qt = (nq + 127) / 128;
  // an even number of query tiles runs as CTA pairs (one cta_group::2 MMA of M = 256 per pair); the grid stays
  // range-major, so two consecutive CTAs (one cluster) are the two query tiles of one pair
  const bool pair = h->gemm_pair != 0 && g->pair_ok && !lite && n_qt % 2 == 0;
  uint32_t ctas = max_ctas ? std::min<uint32_t>(max_ctas, (uint32_t)h->num_sms) : (uint32_t)h->num_sms;
  if (pair) ctas &= ~1u;
  uint32_t n_ranges = ctas / n_qt;
  if (n_ranges < 1) n_ranges = 1;
  const uint32_t n_tiles = (uint32_t)((h->desc.n_docs + kTileDocs - 1) / kTileDocs);
  if (n_ranges > n_tiles) n_ranges = n_tiles;
  if (n_ranges > kMergeMaxLists || (size_t)n_ranges * n_qt * 128 > g->max_lists) return h->fail(OI_ERR_CUDA, "internal: GEMM list workspace too small");
  const uint32_t cap = h->gemm_cap ? (uint32_t)h->gemm_cap : g->cap;
  const uint32_t rows = n_qt * 128;
  {
    const size_t n = (size_t)rows * h->desc.dim / 2;
    unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)h->num_sms * 8);
    gemm_prep_queries_kernel<<<blocks, 256, 0, st>>>(d_queries, nq, rows, h->desc.dim, reinterpret_cast<uint32_t *>(g->d_qb));
    ++h->launches;
    OI_CK(cudaGetLastError());
  }
  // Two passes.  PROBE: every CTA scores `pt` tiles of a strided sample of the shard (about 1/256 of its tiles) and
  // keeps only the maxima of groups of 8 scores; the merge's k-th best of those is a score at least k documents
  // reach, and its k/2-th, k/4-th ... best are the rungs of the ladder.  MAIN: all tiles, filtered by the bound, which
  // climbs the ladder as the grid-wide counters confirm the rungs (a list that still fills up is cut to its best k in
  // the kernel, which raises its own bound), then the exact top-k of what passed.  Shards with only a few tiles per
  // CTA skip the probe: their lists hold everything.
  const uint32_t tiles_per_cta = (n_tiles + n_ranges - 1) / n_ranges;
  const uint32_t pt_max = std::max<uint32_t>(1u, (cap - kTileDocs) / 8u);
  uint32_t pt = h->gemm_sample_tiles > 0 ? (uint32_t)h->gemm_sample_tiles : (tiles_per_cta + 255) / 256;
  pt = std::min(std::max(pt, 1u), pt_max);
  const bool do_probe = !d_dump && (h->gemm_sample_tiles > 0 || tiles_per_cta >= 8);
  const float *thr = nullptr;
  if (do_probe) {
    const uint32_t n_probe = (uint32_t)std::min<uint64_t>((uint64_t)n_ranges * pt, n_tiles);
    const uint32_t stride = n_tiles / n_probe;
    if ((s = gemm_launch(h, nq, n_qt, n_ranges, k, cap, 0, n_probe, stride, true, nullptr, nullptr, lite, pair, st))) return s;
    gemm_merge_kernel<<<nq, 256, 0, st>>>(g->d_cand, g->d_cnt, cap, n_ranges, n_qt, k, nullptr, g->d_keys_a, g->d_lvl_thr, g->d_lvl_cnt);
    ++h->launches;
    OI_CK(cudaGetLastError());
    thr = g->d_lvl_thr;
  }
  if ((s = gemm_launch(h, nq, n_qt, n_ranges, k, cap, 0, n_tiles, 1, false, thr, d_dump, lite, pair, st))) return s;
  gemm_merge_kernel<<<nq, 256, 0, st>>>(g->d_cand, g->d_cnt, cap, n_ranges, n_qt, k, nullptr, d_out_keys, nullptr, nullptr);
  ++h->launches;
  OI_CK(cudaGetLastError());
  return OI_OK;
}
