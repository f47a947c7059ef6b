// bm25.cu — BM25 over a CSR inverted index (docs/SPEC.md §3): index load / on-device synthetic
// build / weight folding, and the doc-range-blocked scoring kernel with the top-k fused in.
//
// Compiled with -fmad=false: SPEC §3 fixes ONE IEEE f32 operation per source-level operation,
// in a fixed order, so that the GPU scores equal the oracle's bit for bit.
//
// Scoring kernel (bm25_blocked_kernel), the hot path of BASELINE config 3:
//   * a work item is (query q, super-range s of documents); items are handed out from an atomic
//     counter, s-major, ~16 per warp, so that the warps running at the same time walk the same part
//     of every posting list (the second reader of a posting finds it in L2) and the last items to
//     finish leave the SMs idle for a small part of the launch.
//   * one WARP owns an item.  It walks its super-range block by block (R = 2048 documents); the
//     block's scores live in shared memory (acc[R] f32), so the dense score vector never exists in HBM.
//   * the query's term table lives in registers (lane l = term l): one ballot finds the lists with
//     postings in the block, one min-reduction the next block with any posting.
//   * per block, the query's DISTINCT terms are applied in ascending term id (SPEC order).  A posting
//     list holds a document at most once, so one term pass has no write conflicts and needs no
//     atomics.  Sparse lists: the first 64-posting chunk of every present list is requested at block
//     start with one bulk copy per list (cp.async.bulk, all in flight at once, per-warp mbarrier).
//     Dense terms (>= 1/16 of the documents) add a weight column, two columns per sweep, and a dense
//     first pass only stores, so the block is never cleared.
//   * after the last term the warp scans acc[] once: every positive score whose key beats the
//     running threshold goes to the warp's candidate buffer (filter + buffer selection, the same
//     scheme as the cosine scan).  A block scanned without any threshold takes the k-th largest of its
//     256 group maxima as a bound first.  The scan is SKIPPED when the threshold exceeds what the
//     query's dense terms can give and no sparse posting of the block produced a score that reaches it.
//   * the item ends with a sorted k-list per (query, super-range); bm25 merge = one CTA per
//     query over the S lists.  A finished item also folds its list into the query's running best-k
//     (per-query try-lock); the k-th key of that list is the grid-wide threshold, so later items of
//     the query filter with the best k of everything scored so far, not of one super-range.
//
//   algorithmic bytes per query = postings touched x 8 B (doc id + folded weight)
#include <cub/device/device_radix_sort.cuh>

#include <algorithm>
#include <cmath>
#include <utility>
#include <vector>

#include "../../include/oi_synth_tables.h"
#include "handle.h"
#include "oi_common.cuh"
#include "oi_postings.cuh"
#include "oi_synth.cuh"

#define OI_BM25_MAX_QTERMS 64
#define OI_BM25_ACC_FLOATS 32768  // 128 KB of block scores per CTA, split over the CTA's groups

struct OiBm25 {
  uint32_t n_terms = 0;
  uint64_t n_postings = 0;
  u64 *d_term_off = nullptr;    // [n_terms + 1]
  uint32_t *d_doc_ids = nullptr;  // [P] shard-local doc ids, ascending inside a list
  uint32_t *d_tfs = nullptr;      // [P]
  uint32_t *d_doc_len = nullptr;  // [n_docs]
  float *d_w = nullptr;           // [P] folded weights (after finalize; export)
  uint2 *d_post = nullptr;        // [P + 68] interleaved (doc id, weight bits): what the scoring kernel streams
  float *d_dense = nullptr;       // [n_dense][dense_stride] weight columns of the densest terms
  int *d_dense_slot = nullptr;    // [n_terms] column index or -1
  float *d_dense_max = nullptr;   // [32] largest weight of each dense column
  uint32_t n_dense = 0, dense_stride = 0;
  bool finalized = false;
  bool attr_set = false;          // dynamic shared-memory limit of the scoring kernels raised
  // search workspace
  uint32_t *d_qterms = nullptr;   // [max_batch][64] sorted distinct valid terms
  uint32_t *d_qnt = nullptr;      // [max_batch]
  u64 *d_gthr = nullptr;          // [max_batch]
  uint32_t *d_counter = nullptr;  // item counter
  u64 *d_lists = nullptr;         // [S][nq][k]
  size_t lists_cap = 0;           // in keys
  u64 *d_best = nullptr;          // [max_batch][max_k] running best k per query (threshold accelerator)
  uint32_t *d_qlock = nullptr;    // [max_batch] try-lock of d_best[q]
  uint32_t *d_in_terms = nullptr; // staging of the host call's flat term array [max_batch * 64]
  uint32_t *d_in_offs = nullptr;  // [max_batch + 1]
};

namespace {

// ------------------------------------------------------------------------------------------------
// group = the threads that own one work item.  One warp: __syncwarp; several warps: named barrier.
// ------------------------------------------------------------------------------------------------
struct Grp {
  int tid;   // thread index inside the group
  int size;  // threads in the group (multiple of 32)
  int bar;   // named barrier id (1..15) for multi-warp groups
  __device__ __forceinline__ void sync() const {
    if (size == 32) __syncwarp();
    else asm volatile("bar.sync %0, %1;" ::"r"(bar), "r"(size) : "memory");
  }
};

__device__ __forceinline__ void grp_bitonic_desc(u64 *buf, uint32_t n, const Grp &g) {
  for (uint32_t k = 2; k <= n; k <<= 1) {
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t i = g.tid; i < (n >> 1); i += g.size) {
        uint32_t l = ((i & ~(j - 1)) << 1) | (i & (j - 1));
        uint32_t r = l | j;
        u64 a = buf[l], b = buf[r];
        bool desc = (l & k) == 0;
        if ((a < b) == desc) { buf[l] = b; buf[r] = a; }
      }
      g.sync();
    }
  }
}

struct GrpCtl {
  u64 thr;        // k-th best key seen by this item so far (0 = none)
  uint32_t cnt;   // candidates in the buffer
  uint32_t item;  // current work item
  uint32_t aux;   // scratch counter (survivor count of a block)
  uint32_t pad;
};

// keeps the best k of buf[0..cnt), sorted descending; raises thr when k are held
__device__ __forceinline__ void grp_compact(u64 *buf, GrpCtl *ctl, uint32_t cap, uint32_t k, const Grp &g) {
  uint32_t c = min(ctl->cnt, cap);
  uint32_t n = oi_next_pow2(c);
  g.sync();
  for (uint32_t i = c + g.tid; i < n; i += g.size) buf[i] = 0ull;
  g.sync();
  grp_bitonic_desc(buf, n, g);
  if (g.tid == 0) {
    uint32_t keep = min(c, k);
    ctl->cnt = keep;
    if (keep == k && buf[k - 1] > ctl->thr) ctl->thr = buf[k - 1];
  }
  g.sync();
}

__device__ __forceinline__ u64 ld_relaxed_u64(const u64 *p) {
  u64 v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

#define OI_BM25_NONE 0xFFFFFFFFu
#define OI_BM25_MAX_DENSE 32
#define OI_BM25_POST_PAD 68  // postings of 0xFF padding after the last list: a 64-posting chunk read from any cursor stays in bounds

struct Bm25Params {
  const u64 *term_off;
  const uint32_t *doc_ids;
  const uint2 *post;          // [P + 68] interleaved (doc id, folded weight bits)
  const float *dense;         // [n_dense][dense_stride] weight columns of the densest terms (0 where absent)
  const int *dense_slot;      // [n_terms] column of a term, or -1
  const float *dense_max;     // [n_dense] largest weight of each column (selection skip, see the kernel)
  uint32_t dense_stride;
  const uint32_t *qterms;     // [nq][64]
  const uint32_t *qnt;        // [nq]
  u64 *gthr;                  // [nq]
  uint32_t *counter;
  u64 *lists;                 // [S][nq][k]
  u64 *best;                  // [nq][k] running best k of each query's finished items (threshold accelerator; zeroed by prep)
  uint32_t *qlock;            // [nq] one try-lock per query for folding an item into best[]
  uint32_t n_docs, doc_base, nq, k;
  uint32_t cap;               // candidate buffer keys per warp (power of two, >= 2k)
  uint32_t R;                 // docs per block (a power of two)
  uint32_t r_shift;           // log2(R)
  uint32_t J;                 // blocks per super-range
  uint32_t S;                 // super-ranges
  uint32_t n_blocks;
  uint32_t ng;                // warps (= work items in flight) per CTA
  uint32_t nslot;             // staged 64-posting chunks per warp (0 = no staging)
  uint32_t cold_bound;        // 1: k <= 256 and the staging buffer can hold 256 group maxima (cold-start bound)
};

__device__ __forceinline__ uint4 ldg_post2(const uint2 *p) {
  return __ldg(reinterpret_cast<const uint4 *>(p));
}

// One term's postings inside the block [bbase, bend): the warp reads the interleaved (doc, weight) array 64
// postings at a time (one 16-byte load = 2 postings per lane) from the 16-byte-aligned pair at or below the
// cursor, adds every weight whose document is below `bend` to acc[], and stops at the first posting outside
// the block.  *pos_out = the new cursor, *nxt_out = the document there (NONE at the end of the list).
// `st` (warp-uniform, may be NULL) = this warp's staged copy of the first chunk: lane l's 16 bytes at st[l],
// a bulk copy of the 512 bytes from exactly the address the first iteration would load.
__device__ __forceinline__ void sparse_pass(const uint2 *__restrict__ post, u64 base, uint32_t pos, uint32_t end, uint32_t bbase,
                                            uint32_t bend, float *acc, int lane, const uint4 *st, uint32_t *pos_out,
                                            uint32_t *nxt_out, float &mx) {
  // list-local 32-bit slot numbers over a 16-byte-aligned view of the list: slot j = posting (j - par)
  const uint32_t par = (uint32_t)(base & 1ull);
  const uint2 *lp = post + (base - par);
  const uint32_t j0 = pos + par, jend = end + par;  // [j0, jend) = the postings still to consume
  uint32_t a = j0 & ~1u;
  uint32_t skip = j0 - a;  // a leading slot below the cursor (0 or 1)
  uint32_t applied = 0, nxt = OI_BM25_NONE;
  for (;;) {
    const uint32_t idx = a + 2u * (uint32_t)lane;
    uint4 v = make_uint4(OI_BM25_NONE, 0u, OI_BM25_NONE, 0u);
    if (idx < jend) v = st ? st[lane] : ldg_post2(lp + idx);  // the array is padded: reading the pair is in bounds
    st = nullptr;
    if (idx + 1 >= jend) v.z = OI_BM25_NONE;      // second slot belongs to the next list
    if (idx < j0) v.x = OI_BM25_NONE;             // leading slot below the cursor: skipped, not applied
    const bool in0 = v.x < bend, in1 = v.z < bend;
    if (in0) {
      float *x = acc + (v.x - bbase);
      const float nx = *x + __uint_as_float(v.y);  // SPEC §3: one f32 add, previous terms first
      *x = nx;
      mx = fmaxf(mx, nx);
    }
    if (in1) {
      float *x = acc + (v.z - bbase);
      const float nx = *x + __uint_as_float(v.w);
      *x = nx;
      mx = fmaxf(mx, nx);
    }
    const uint32_t n = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, in0)) + (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, in1));
    applied += n;
    if (skip + n < 64u) {  // slot (skip + n) is the first posting outside the block, or past the end of the list
      const uint32_t sl = skip + n;
      const uint32_t d = (sl & 1u) ? v.z : v.x;
      nxt = __shfl_sync(0xFFFFFFFFu, d, (int)(sl >> 1));
      if (a + sl >= jend) nxt = OI_BM25_NONE;
      break;
    }
    a += 64;
    skip = 0;
  }
  *pos_out = pos + applied;
  *nxt_out = nxt;
}

// Dense terms: the weight column of the block is added to every document (0.0f where the term is absent, which
// leaves a non-negative f32 sum bit-for-bit unchanged) with 128-bit loads; see block_passes.

// One lane's share of the work item's term table: lane l of set 0 holds term l of the query (ascending term id),
// lane l of set 1 holds term 32 + l.  Keeping the cursors in registers (instead of shared-memory arrays every lane
// re-reads per term and per block) makes "which lists have postings in this block" one ballot, "next block with
// any posting" one warp reduction, and lets the warp visit only the lists that are present.
struct TermRegs {
  u64 base;       // posting-array offset of the list
  uint32_t cur;   // postings consumed so far
  uint32_t end;   // list length
  uint32_t nxt;   // document at the cursor (NONE = exhausted / no such term)
  uint32_t den;   // dense column of the term (NONE = sparse)
};

__device__ __forceinline__ void term_setup(TermRegs &T, const Bm25Params &p, uint32_t q, uint32_t i, uint32_t nt, uint32_t doc0) {
  T.base = 0; T.cur = 0; T.end = 0; T.nxt = OI_BM25_NONE; T.den = OI_BM25_NONE;
  if (i >= nt) return;
  const uint32_t t = p.qterms[(size_t)q * OI_BM25_MAX_QTERMS + i];
  const u64 lo = p.term_off[t], hi = p.term_off[t + 1];
  const int slot = p.dense_slot[t];
  T.base = lo;
  T.end = (uint32_t)(hi - lo);
  if (slot >= 0) {  // dense terms touch every block
    T.den = (uint32_t)slot;
    T.nxt = doc0;
  } else {          // one binary search positions the cursor at the super-range start
    u64 a = lo, b = doc0 ? hi : lo;  // nothing precedes the shard's first document
    while (a < b) {
      const u64 mid = a + ((b - a) >> 1);
      if (__ldg(p.doc_ids + mid) < doc0) a = mid + 1; else b = mid;
    }
    T.cur = (uint32_t)(a - lo);
    T.nxt = a < hi ? __ldg(p.doc_ids + a) : OI_BM25_NONE;
  }
}

// global -> shared bulk copy (TMA 1-D, SASS UBLKCP) without a cache hint: postings are re-read by the other queries
__device__ __forceinline__ void bm25_bulk_g2s(void *smem_dst, const void *gmem_src, uint32_t bytes, void *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(oi_smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(oi_smem_u32(bar))
               : "memory");
}

// Two IEEE f32 additions in one instruction (add.rn.f32x2, SASS FADD2): bit for bit what two add.rn.f32 give, half
// the issue slots of the dense sweeps.
__device__ __forceinline__ void add2(float &a0, float &a1, float b0, float b1) {
  unsigned long long x, y;
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(y) : "f"(b0), "f"(b1));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(x) : "l"(x), "l"(y));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(a0), "=f"(a1) : "l"(x));
}
__device__ __forceinline__ void add4(float4 &a, const float4 &b) {
  add2(a.x, a.y, b.x, b.y);
  add2(a.z, a.w, b.z, b.w);
}

// One or two dense columns in one sweep over the block's scores: x = (FRESH ? 0 : acc) + a (+ b), ascending term
// order, software-pipelined in stages of 2 x 128 bits per column and lane.  FRESH = no pass has written acc[] for this block yet: the
// sweep then only stores (0.0f + w == w for every weight, bit for bit), so the block needs no clearing pass.
template <bool FRESH, int NC>
__device__ __forceinline__ void dense_stage_load(const float4 *__restrict__ c0, const float4 *__restrict__ c1, uint32_t j, int lane, float4 (&va)[2],
                                                 float4 (&vb)[2]) {
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    va[u] = __ldg(c0 + j + 32 * u + lane);
    if (NC == 2) vb[u] = __ldg(c1 + j + 32 * u + lane);
  }
}
template <bool FRESH, int NC>
__device__ __forceinline__ void dense_stage_apply(float4 *a4, uint32_t j, int lane, const float4 (&va)[2], const float4 (&vb)[2]) {
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    float4 x = va[u];
    if (!FRESH) {
      float4 o = a4[j + 32 * u + lane];
      add4(o, x);  // o + x: the earlier terms' sum first
      x = o;
    }
    if (NC == 2) add4(x, vb[u]);
    a4[j + 32 * u + lane] = x;
  }
}

template <bool FRESH, int NC>
__device__ __forceinline__ void dense_sweep(const float4 *__restrict__ c0, const float4 *__restrict__ c1, float4 *a4, uint32_t R, int lane) {
  // software pipeline over stages of 2 x 128 bits per column and lane: the loads of stage t + 1 are in flight while
  // stage t is added and stored, so a sweep exposes one L2 latency instead of one per group of loads
  float4 va0[2], vb0[2], va1[2], vb1[2];
  dense_stage_load<FRESH, NC>(c0, c1, 0, lane, va0, vb0);
  for (uint32_t j0 = 0; j0 < R / 4; j0 += 128) {
    dense_stage_load<FRESH, NC>(c0, c1, j0 + 64, lane, va1, vb1);
    dense_stage_apply<FRESH, NC>(a4, j0, lane, va0, vb0);
    if (j0 + 128 < R / 4) dense_stage_load<FRESH, NC>(c0, c1, j0 + 128, lane, va0, vb0);
    dense_stage_apply<FRESH, NC>(a4, j0 + 64, lane, va1, vb1);
  }
}

// The term passes of one block for one register set, ascending term id (SPEC §3 order).  First every sparse list
// with postings in the block gets its first 64-posting chunk requested -- lane i issues ONE bulk copy for term i,
// all lists in flight at once, completion counted on the warp's mbarrier -- then the present lists are visited
// in order: dense terms add their columns (two consecutive ones share a sweep), a sparse term consumes its chunk
// (staged, or loaded directly when the warp's staging slots are taken) with ONE shuffle of set-up -- the owner lane
// packs "postings left in the list from the chunk's first slot" and the 0/1 leading slot below the cursor into one
// word -- and only a segment longer than the chunk fetches the rest of the list's registers and goes on with the
// general loop (sparse_pass).  `fresh` = acc[] holds nothing for this block yet: a dense first pass overwrites it, a
// sparse first pass clears it first.  `touched` accumulates an upper bound of the documents with a positive score
// (postings applied; R per dense sweep); `mx` = per lane, the largest score a sparse posting produced.
template <uint32_t RT>
__device__ __forceinline__ void block_passes(TermRegs &T, uint32_t dmask, const Bm25Params &p, float *acc, uint4 *stage, void *mbar,
                                             uint32_t &phase, bool &fresh, uint32_t &touched, float &mx, uint32_t bbase, uint32_t bend,
                                             int lane) {
  const uint32_t R = RT ? RT : p.R;
  const uint32_t pm = __ballot_sync(0xFFFFFFFFu, T.nxt < bend);
  if (pm == 0) return;
  const uint32_t sm = pm & ~dmask;
  // chunk geometry of this lane's list: 16-byte-aligned pair at or below the cursor
  const uint32_t par = (uint32_t)(T.base & 1ull);
  const uint32_t ca = (T.cur + par) & ~1u;
  const u64 coff = (T.base - par) + ca;                                   // posting-array index of the chunk's slot 0
  const uint32_t meta = (min(T.end + par - ca, 1u << 20) << 1) | ((T.cur + par) - ca);  // (slots left << 1) | leading slot
  const uint32_t n_staged = min((uint32_t)__popc(sm), p.nslot);
  if (n_staged) {
    if (lane == 0) oi_mbar_expect_tx(mbar, n_staged * 512u);
    const uint32_t my_slot = (uint32_t)__popc(sm & ((1u << lane) - 1u));
    if (((sm >> lane) & 1u) && my_slot < p.nslot)
      bm25_bulk_g2s(stage + my_slot * 32u, p.post + coff, 512u, mbar);  // the array is padded by 64 postings
  }
  float4 *a4 = reinterpret_cast<float4 *>(acc);
  const uint32_t nxt_dense = bend < p.n_docs ? bend : OI_BM25_NONE;  // a dense term is present in every block
  bool waited = false;
  uint32_t m = pm;
  uint32_t slot = 0;  // sparse lists visited so far = staging slot of the next one
  while (m) {
    const int i = __ffs((int)m) - 1;
    m &= m - 1u;
    if ((dmask >> i) & 1u) {
      const uint32_t den = __shfl_sync(0xFFFFFFFFu, T.den, i);
      const float4 *c0 = reinterpret_cast<const float4 *>(p.dense + (size_t)den * p.dense_stride + bbase);
      int i2 = -1;
      if (m) {
        const int cand = __ffs((int)m) - 1;
        if ((dmask >> cand) & 1u) i2 = cand;  // the next present term is dense too: one sweep adds both columns
      }
      if (i2 >= 0) {
        m &= m - 1u;
        const uint32_t den2 = __shfl_sync(0xFFFFFFFFu, T.den, i2);
        const float4 *c1 = reinterpret_cast<const float4 *>(p.dense + (size_t)den2 * p.dense_stride + bbase);
        if (fresh) dense_sweep<true, 2>(c0, c1, a4, R, lane);
        else dense_sweep<false, 2>(c0, c1, a4, R, lane);
      } else {
        if (fresh) dense_sweep<true, 1>(c0, c0, a4, R, lane);
        else dense_sweep<false, 1>(c0, c0, a4, R, lane);
      }
      fresh = false;
      touched += R;
      if (lane == i || lane == i2) T.nxt = nxt_dense;
    } else {
      if (fresh) {  // a sparse first pass scatters into the block: clear it first
        const float4 zero4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll 4
        for (uint32_t j = lane; j < R / 4; j += 32) a4[j] = zero4;
        fresh = false;
        __syncwarp();
      }
      const uint32_t mt = __shfl_sync(0xFFFFFFFFu, meta, i);
      const uint32_t skip = mt & 1u, rem = mt >> 1;
      const uint32_t idx = 2u * (uint32_t)lane;
      uint4 v = make_uint4(OI_BM25_NONE, 0u, OI_BM25_NONE, 0u);
      if (slot < n_staged) {
        if (!waited) { oi_mbar_wait(mbar, phase); phase ^= 1u; waited = true; }
        v = stage[slot * 32u + lane];
      } else {
        const u64 off = __shfl_sync(0xFFFFFFFFu, coff, i);
        if (idx < rem) v = ldg_post2(p.post + off + idx);  // the array is padded: reading the pair is in bounds
      }
      ++slot;
      if (idx + 1 >= rem) v.z = OI_BM25_NONE;             // second slot belongs to the next list
      if (idx >= rem || idx < skip) v.x = OI_BM25_NONE;   // past the list / the leading slot below the cursor
      const bool in0 = v.x < bend, in1 = v.z < bend;
      if (in0) {
        float *x = acc + (v.x - bbase);
        const float nx = *x + __uint_as_float(v.y);  // SPEC §3: one f32 add, previous terms first
        *x = nx;
        mx = fmaxf(mx, nx);
      }
      if (in1) {
        float *x = acc + (v.z - bbase);
        const float nx = *x + __uint_as_float(v.w);
        *x = nx;
        mx = fmaxf(mx, nx);
      }
      const uint32_t n = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, in0)) + (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, in1));
      const uint32_t sl = skip + n;  // first slot outside the block (or past the end of the list: masked to NONE above)
      if (sl < 64u) {
        const uint32_t nxt = __shfl_sync(0xFFFFFFFFu, (sl & 1u) ? v.z : v.x, (int)(sl >> 1));
        touched += n;
        if (lane == i) { T.cur += n; T.nxt = nxt; }
      } else {  // the segment is longer than the chunk: go on with direct loads
        const u64 base = __shfl_sync(0xFFFFFFFFu, T.base, i);
        const uint32_t cur = __shfl_sync(0xFFFFFFFFu, T.cur, i);
        const uint32_t end = __shfl_sync(0xFFFFFFFFu, T.end, i);
        uint32_t pos_new, nxt;
        sparse_pass(p.post, base, cur + n, end, bbase, bend, acc, lane, nullptr, &pos_new, &nxt, mx);
        touched += pos_new - cur;
        if (lane == i) { T.cur = pos_new; T.nxt = nxt; }
      }
    }
    __syncwarp();  // the next pass may touch the same documents
  }
}

// Compile-time instrumentation (not in the shipped build): -DOI_BM25_STATS counts, per launch, the (query, block) pairs
// scored, those whose threshold exceeds the dense bound, those that skip the selection sweep and those scored without
// any threshold, and prints them after the launch (profiles/r02_ncu_bm25.md); -DOI_BM25_NOSKIP disables the skip (A/B).
#ifdef OI_BM25_STATS
__device__ unsigned long long g_bm25_stats[4];  // blocks scored, threshold above the dense bound, selection skipped, no threshold
__global__ void bm25_stats_print_kernel() {
  printf("bm25 stats: blocks %llu, thr > dense_ub %llu, skipped %llu, cold %llu\n", g_bm25_stats[0], g_bm25_stats[1], g_bm25_stats[2], g_bm25_stats[3]);
  g_bm25_stats[0] = g_bm25_stats[1] = g_bm25_stats[2] = g_bm25_stats[3] = 0ull;
}
#endif

// dynamic shared memory layout (per CTA, NG = warps per CTA):
//   float  acc[NG][R]               block scores
//   u64    cand[NG][cap]            candidate buffers
//   uint4  stage[NG][nslot][32]     staged first chunks (64 postings each) of the block's sparse lists
//   GrpCtl ctl[NG]
//   u64    mbar[NG]                 one mbarrier per warp for its bulk copies
template <int MAXT, uint32_t RT>  // RT = documents per block at compile time (0 = p.R)
__global__ void __launch_bounds__(MAXT, 1) bm25_blocked_kernel(const Bm25Params p) {
  extern __shared__ __align__(16) unsigned char s_dyn[];
  const int NG = (int)p.ng;
  const int gi = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Grp g;
  g.tid = lane;
  g.size = 32;
  g.bar = 0;

  const uint32_t R = RT ? RT : p.R;
  float *acc = reinterpret_cast<float *>(s_dyn) + (size_t)gi * R;
  u64 *cand_all = reinterpret_cast<u64 *>(s_dyn + sizeof(float) * (size_t)NG * R);
  u64 *cand = cand_all + (size_t)gi * p.cap;
  uint4 *stage_all = reinterpret_cast<uint4 *>(cand_all + (size_t)NG * p.cap);
  uint4 *stage = stage_all + (size_t)gi * p.nslot * 32;
  GrpCtl *ctl_all = reinterpret_cast<GrpCtl *>(stage_all + (size_t)NG * p.nslot * 32);
  GrpCtl *ctl = ctl_all + gi;
  u64 *mbar = reinterpret_cast<u64 *>(ctl_all + NG) + gi;  // NG x 24 bytes of control blocks keep 8-byte alignment

  if (lane == 0) {
    oi_mbar_init(mbar, 1);
    oi_mbar_fence_init();
  }
  __syncwarp();
  uint32_t phase = 0;
  const uint32_t n_items = p.S * p.nq;
  const uint32_t k = p.k, cap = p.cap;

  for (;;) {
    __syncwarp();
    uint32_t item = 0;
    if (lane == 0) item = atomicAdd(p.counter, 1u);
    item = __shfl_sync(0xFFFFFFFFu, item, 0);
    if (item >= n_items) break;
    const uint32_t s = item / p.nq, q = item % p.nq;
    const uint32_t nt = p.qnt[q];
    const uint32_t blk0 = s * p.J, blk1 = min(p.n_blocks, blk0 + p.J);
    const uint32_t doc0 = blk0 * R;

    // ---- item set-up: lane l takes terms l and 32 + l of the query
    TermRegs T0, T1;
    term_setup(T0, p, q, (uint32_t)lane, nt, doc0);
    term_setup(T1, p, q, 32u + (uint32_t)lane, nt, doc0);
    if (lane == 0) { ctl->cnt = 0; ctl->thr = 0ull; ctl->aux = 0; }
    const uint32_t dm0 = __ballot_sync(0xFFFFFFFFu, T0.den != OI_BM25_NONE);
    const uint32_t dm1 = __ballot_sync(0xFFFFFFFFu, T1.den != OI_BM25_NONE);
    // no document can get more than `dense_ub` from the query's dense terms: the sum of the columns' largest weights
    // (any association; the factor covers the rounding difference to the SPEC-order sum of a real document)
    float dense_ub = (T0.den != OI_BM25_NONE ? __ldg(p.dense_max + T0.den) : 0.0f) + (T1.den != OI_BM25_NONE ? __ldg(p.dense_max + T1.den) : 0.0f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) dense_ub += __shfl_xor_sync(0xFFFFFFFFu, dense_ub, o);
    dense_ub *= 1.0001f;
#ifdef OI_BM25_NOSKIP
    dense_ub = 3.0e38f;
#endif
    __syncwarp();

    uint32_t blk = blk0;
    while (blk < blk1) {
      // ---- skip straight to the next block that holds a posting of any query term -------------
      const uint32_t mn = __reduce_min_sync(0xFFFFFFFFu, min(T0.nxt, T1.nxt));
      if (mn == OI_BM25_NONE) break;
      blk = max(blk, mn >> p.r_shift);
      if (blk >= blk1) break;
      const uint32_t bbase = blk * R;
      const uint32_t bend = min(p.n_docs, bbase + R);
      ++blk;
      // the grid-wide threshold is requested now and consumed after the passes
      const u64 gthr_now = ld_relaxed_u64(p.gthr + q);
      bool fresh = true;  // acc[] holds the previous block's scores until the first pass overwrites or clears it
      uint32_t touched = 0;
      float mx = 0.0f;
      block_passes<RT>(T0, dm0, p, acc, stage, mbar, phase, fresh, touched, mx, bbase, bend, lane);
      if (nt > 32) block_passes<RT>(T1, dm1, p, acc, stage, mbar, phase, fresh, touched, mx, bbase, bend, lane);
      // ---- selection: positive scores that beat the running threshold -------------------------
      const u64 thr = max(ctl->thr, gthr_now);
      float tsc = thr ? oi_key_score(thr) : 0.0f;  // a survivor has score >= tsc (and > 0)
      __syncwarp();
      // Once the threshold exceeds what the dense terms alone can give, a survivor must hold a sparse posting, and
      // the sparse passes saw every such document's score as it grew (weights are >= 0, so a score that ends at or
      // above the threshold was at or above it in the last pass that touched it): no lane saw one -> nothing to
      // select, and the sweep over the block's 2048 scores -- a fifth of the kernel's instructions -- is skipped.
#ifdef OI_BM25_STATS
      if (lane == 0) {
        atomicAdd(&g_bm25_stats[0], 1ull);
        if (tsc > dense_ub) atomicAdd(&g_bm25_stats[1], 1ull);
        if (thr == 0ull) atomicAdd(&g_bm25_stats[3], 1ull);
      }
      if (tsc > dense_ub && !__any_sync(0xFFFFFFFFu, mx >= tsc)) {
        if (lane == 0) atomicAdd(&g_bm25_stats[2], 1ull);
        continue;
      }
#else
      if (tsc > dense_ub && !__any_sync(0xFFFFFFFFu, mx >= tsc)) continue;
#endif
      if (thr == 0ull && p.cold_bound && touched + ctl->cnt > cap) {
        // cold start (no threshold yet: the first block of an item whose query has none either, i.e. every block of a
        // single-query call) and more positive scores than the buffer can take: without a bound every one of them
        // is a candidate and the buffer is sorted a dozen times.  The k-th largest of the block's 256 group maxima (groups of R / 256 documents) is a score at
        // least k documents of the block reach, so nothing below it can be in the top k: one sort of 256 values
        // replaces the repeated compactions.  The staging buffer is idle here and serves as scratch.
        uint32_t *gm = reinterpret_cast<uint32_t *>(stage);
        const float4 *accr = reinterpret_cast<const float4 *>(acc);
        const uint32_t per_group = R / 1024u;  // float4s per group and lane: lane l owns float4s l, l + 32, ...
#pragma unroll
        for (uint32_t gi8 = 0; gi8 < 8; ++gi8) {
          float mx = 0.0f;
          for (uint32_t u = 0; u < per_group; ++u) {
            const float4 v = accr[(gi8 * per_group + u) * 32u + lane];
            mx = fmaxf(mx, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
          }
          gm[gi8 * 32u + lane] = __float_as_uint(mx);  // scores are >= 0: the bit patterns order like the values
        }
        __syncwarp();
        for (uint32_t k2 = 2; k2 <= 256u; k2 <<= 1) {
          for (uint32_t j = k2 >> 1; j > 0; j >>= 1) {
#pragma unroll
            for (uint32_t i = lane; i < 128u; i += 32) {
              const uint32_t l = ((i & ~(j - 1)) << 1) | (i & (j - 1));
              const uint32_t r = l | j;
              const uint32_t a = gm[l], b = gm[r];
              const bool desc = (l & k2) == 0;
              if ((a < b) == desc) { gm[l] = b; gm[r] = a; }
            }
            __syncwarp();
          }
        }
        tsc = __uint_as_float(gm[k - 1]);
        __syncwarp();
        // the scratch was written through the generic proxy; the next block's bulk copies write it through the async one
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      }
      // one pass reads and tests the block, 4 x 128 bits per lane per step (the next block's first pass overwrites
      // or clears acc[]).  In steady state only a handful of scores survive the threshold; a group with a survivor
      // that finds the buffer full is rewritten with only the scores still to be ranked, for the overflow path.
      float4 *accw = reinterpret_cast<float4 *>(acc);
#pragma unroll 2
      for (uint32_t jb = 0; jb < R / 4; jb += 128) {
        float4 vv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) vv[u] = accw[jb + 32 * u + lane];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float4 v = vv[u];
          const float m4 = fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w));
          if (m4 > 0.0f && m4 >= tsc) {
            const uint32_t j = jb + 32 * u + lane;
            const float sc4[4] = {v.x, v.y, v.z, v.w};
            float back[4] = {0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
            for (int c4 = 0; c4 < 4; ++c4) {
              if (sc4[c4] > 0.0f && sc4[c4] >= tsc) {
                const u64 key = oi_make_key(sc4[c4], p.doc_base + bbase + 4 * j + c4);
                if (key > thr) {
                  const uint32_t at = atomicAdd(&ctl->cnt, 1u);
                  if (at < cap) cand[at] = key;
                  else back[c4] = sc4[c4];
                }
              }
            }
            accw[j] = make_float4(back[0], back[1], back[2], back[3]);  // only the scores that did not fit stay
          }
        }
      }
      __syncwarp();
      if (ctl->cnt > cap) {
        // overflow (cold threshold): the buffer holds `cap` valid keys; of the scores that can still matter, acc[]
        // holds exactly those that did not fit (everything else left there is below the threshold and fails the
        // key test again); rank them in spans that cannot overflow the buffer, compacting between spans
        __syncwarp();
        if (lane == 0) ctl->cnt = cap;
        __syncwarp();
        grp_compact(cand, ctl, cap, k, g);
        if (lane == 0 && ctl->cnt == k) atomicMax(p.gthr + q, ctl->thr);
        const uint32_t span_all = bend - bbase;
        uint32_t b0 = 0;
        while (b0 < span_all) {
          const uint32_t span = min(span_all - b0, cap - ctl->cnt);
          const u64 t2 = max(thr, ctl->thr);
          __syncwarp();
          for (uint32_t j = b0 + lane; j < b0 + span; j += 32) {
            const float sc = acc[j];
            if (sc > 0.0f) {
              const u64 key = oi_make_key(sc, p.doc_base + bbase + j);
              if (key > t2) { const uint32_t at = atomicAdd(&ctl->cnt, 1u); if (at < cap) cand[at] = key; }
            }
          }
          b0 += span;
          __syncwarp();
          if (ctl->cnt > cap / 2) {
            grp_compact(cand, ctl, cap, k, g);
            if (lane == 0 && ctl->cnt == k) atomicMax(p.gthr + q, ctl->thr);
          }
        }
      } else if (ctl->cnt > cap / 2) {
        grp_compact(cand, ctl, cap, k, g);
        if (lane == 0 && ctl->cnt == k) atomicMax(p.gthr + q, ctl->thr);
      }
      __syncwarp();
    }
    // ---- item done: publish the sorted list, and fold it into the query's running best-k ----------
    grp_compact(cand, ctl, cap, k, g);
    if (lane == 0 && ctl->cnt == k) atomicMax(p.gthr + q, ctl->thr);
    u64 *out = p.lists + ((size_t)s * p.nq + q) * k;
    const uint32_t cnt = ctl->cnt;  // <= k, and 2k <= cap
    for (uint32_t i = lane; i < k; i += 32) out[i] = i < cnt ? cand[i] : 0ull;
    // best[q][0..k) = the best k keys of the items of query q folded in so far (sorted, 0 = empty); its k-th key is
    // published as the grid-wide threshold.  An item's own k-th best only bounds the documents of its super-range;
    // the folded list bounds everything scored so far, so the items that start later filter with (nearly) the final
    // threshold: the survivors of a query fall from ~k per item to ~k ln(items) in all and most blocks skip the
    // selection sweep.  It only accelerates -- the result is still the merge of the per-item lists -- so an item
    // that finds the list locked (queries of rare terms finish their items in bursts) or has nothing above the
    // current threshold simply does not contribute.
    if (cnt && cand[0] > ld_relaxed_u64(p.gthr + q)) {
      uint32_t got = 0;
      if (lane == 0) {
        got = atomicCAS(p.qlock + q, 0u, 1u) == 0u;
        if (got) __threadfence();
      }
      if (__shfl_sync(0xFFFFFFFFu, got, 0)) {
        // two sorted lists of distinct keys: the merged rank of a key is its index plus the number of keys of the
        // other list above it (one binary search each; no sort, the lock is held for a microsecond)
        u64 *best = p.best + (size_t)q * k;
        u64 *sb = cand + cap / 2;  // cnt <= k <= cap / 2: room for a copy of the running list next to the item's own
        for (uint32_t i = lane; i < k; i += 32) sb[i] = __ldcg(best + i);
        __syncwarp();
        u64 kth = 0ull;  // the key that ends at rank k - 1
        for (uint32_t i = lane; i < k; i += 32) {
          const u64 bk = sb[i];
          if (bk == 0ull) continue;  // empty slots stay empty unless an own key lands there
          uint32_t lo = 0, hi = cnt;
          while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (cand[mid] > bk) lo = mid + 1; else hi = mid;
          }
          const uint32_t r = i + lo;
          if (lo && r < k) __stcg(best + r, bk);
          if (r == k - 1) kth = bk;
        }
        for (uint32_t i = lane; i < cnt; i += 32) {
          const u64 ok = cand[i];
          uint32_t lo = 0, hi = k;
          while (lo < hi) {
            const uint32_t mid = (lo + hi) >> 1;
            if (sb[mid] > ok) lo = mid + 1; else hi = mid;
          }
          const uint32_t r = i + lo;
          if (r < k) __stcg(best + r, ok);
          if (r == k - 1) kth = ok;
        }
        __threadfence();
        if (kth) atomicMax(p.gthr + q, kth);  // exactly one key lands at rank k - 1, if the list is full
        __syncwarp();
        if (lane == 0) atomicExch(p.qlock + q, 0u);
      }
    }
  }
}

// Query preparation, one warp per query: de-duplicates the raw term ids in first-seen order, drops unknown terms and
// empty lists, keeps at most the first 64 distinct known terms (SPEC §3) and writes them in ascending term id.  A
// query may carry any number of raw ids (the host-buffer and the `_dev` entry points behave alike); the usual 8-term
// query is one 32-id chunk: all list-length loads in flight at once, then ranks by counting.
__global__ void __launch_bounds__(128) bm25_prep_queries_kernel(const uint32_t *q_terms, const uint32_t *q_offs, uint32_t nq,
                                                               const u64 *term_off, uint32_t n_terms, uint32_t *out_terms,
                                                               uint32_t *out_nt, u64 *gthr, uint32_t *counter, u64 *best,
                                                               uint32_t k, uint32_t *qlock) {
  __shared__ uint32_t s_kept[4][OI_BM25_MAX_QTERMS];
  const uint32_t q = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  uint32_t *kept = s_kept[threadIdx.x >> 5];
  if (blockIdx.x == 0 && threadIdx.x == 0) *counter = 0;
  if (q >= nq) return;  // warp-uniform
  if (lane == 0) { gthr[q] = 0ull; qlock[q] = 0u; }
  for (uint32_t i = lane; i < k; i += 32) best[(size_t)q * k + i] = 0ull;
  const uint32_t lo = q_offs[q];
  const uint32_t n_in = q_offs[q + 1] - lo;
  uint32_t n_kept = 0;
  for (uint32_t c0 = 0; c0 < n_in && n_kept < OI_BM25_MAX_QTERMS; c0 += 32) {
    const uint32_t i = c0 + (uint32_t)lane;
    const uint32_t t = i < n_in ? q_terms[lo + i] : 0xFFFFFFFFu;
    bool ok = i < n_in && t < n_terms;
    if (ok) ok = term_off[t + 1] != term_off[t];
    for (uint32_t j = 0; j < n_kept; ++j)  // already kept by an earlier chunk
      if (kept[j] == t) ok = false;
    const uint32_t same = __match_any_sync(0xFFFFFFFFu, t);
    const bool first = ok && (same & ((1u << lane) - 1u)) == 0u;  // first occurrence inside the chunk
    const uint32_t fm = __ballot_sync(0xFFFFFFFFu, first);
    const uint32_t pos = n_kept + (uint32_t)__popc(fm & ((1u << lane) - 1u));
    if (first && pos < OI_BM25_MAX_QTERMS) kept[pos] = t;
    n_kept = min((uint32_t)OI_BM25_MAX_QTERMS, n_kept + (uint32_t)__popc(fm));
    __syncwarp();
  }
  // rank = number of kept terms below mine
  uint32_t *o = out_terms + (size_t)q * OI_BM25_MAX_QTERMS;
#pragma unroll
  for (int hh = 0; hh < 2; ++hh) {
    const uint32_t i = (uint32_t)lane + 32u * hh;
    if (i < n_kept) {
      const uint32_t t = kept[i];
      uint32_t rank = 0;
      for (uint32_t j = 0; j < n_kept; ++j) rank += kept[j] < t;
      o[rank] = t;
    }
  }
  if (lane == 0) out_nt[q] = n_kept;
}

// the term of each posting: the warp-tile walk of oi_postings.cuh (bm25_tile_terms / bm25_term_of)

// per-posting folded weight, SPEC §3 association, one IEEE op per line (file built with -fmad=false)
__global__ void __launch_bounds__(256) bm25_weights_kernel(const u64 *term_off, const uint32_t *doc_ids, const uint32_t *tfs,
                                    const uint32_t *doc_len, const float *idf, uint32_t n_terms, u64 n_postings,
                                    float k1, float b, float avgdl, float *w, uint2 *post, const int *dense_slot, float *dense,
                                    uint32_t dense_stride) {
  const float one_minus_b = 1.0f - b;
  const float k1p1 = k1 + 1.0f;
  const int lane = threadIdx.x & 31;
  const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 tile = warp * OI_BM25_TILE; tile < n_postings; tile += n_warps * OI_BM25_TILE) {
    const TileTerms tt = bm25_tile_terms(term_off, n_terms, tile, n_postings, lane);
    uint32_t lo = tt.lo;
    for (uint32_t u = 0; u < OI_BM25_TILE / 32; ++u) {
      const u64 p = tile + 32u * u + (uint32_t)lane;
      if (p >= n_postings) break;
      lo = bm25_term_of(term_off, lo, tt.hi, p);
      const float dl = (float)doc_len[doc_ids[p]];
      const float ratio = dl / avgdl;
      const float bt = b * ratio;
      const float uu = one_minus_b + bt;
      const float norm = k1 * uu;
      const float tf = (float)tfs[p];
      const float num = tf * k1p1;
      const float den = tf + norm;
      const float qv = num / den;
      const float wv = idf[lo] * qv;
      w[p] = wv;
      post[p] = make_uint2(doc_ids[p], __float_as_uint(wv));
      const int slot = dense_slot[lo];
      if (slot >= 0) dense[(size_t)slot * dense_stride + doc_ids[p]] = wv;
    }
  }
}

// largest weight of every dense column (weights are >= 0: the bit patterns order like the values)
__global__ void __launch_bounds__(256) bm25_dense_max_kernel(const float *dense, uint32_t dense_stride, uint32_t n_docs, uint32_t *out_bits) {
  const float *col = dense + (size_t)blockIdx.y * dense_stride;
  float m = 0.0f;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n_docs; i += gridDim.x * blockDim.x) m = fmaxf(m, col[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax(out_bits + blockIdx.y, __float_as_uint(m));
}

// CSR validation on the device (oi_index_load_bm25): every doc id inside the shard, strictly ascending inside a list.
// *err = the smallest offending posting index << 1 | kind (0 = doc id outside the shard, 1 = not ascending); ~0 = none.
__global__ void __launch_bounds__(256) bm25_validate_kernel(const u64 *term_off, const uint32_t *doc_ids, uint32_t n_terms, u64 n_postings,
                                                            uint32_t n_docs, u64 *err) {
  const int lane = threadIdx.x & 31;
  const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 tile = warp * OI_BM25_TILE; tile < n_postings; tile += n_warps * OI_BM25_TILE) {
    const TileTerms tt = bm25_tile_terms(term_off, n_terms, tile, n_postings, lane);
    uint32_t lo = tt.lo;
    for (uint32_t u = 0; u < OI_BM25_TILE / 32; ++u) {
      const u64 p = tile + 32u * u + (uint32_t)lane;
      if (p >= n_postings) break;
      lo = bm25_term_of(term_off, lo, tt.hi, p);
      const uint32_t d = doc_ids[p];
      if (d >= n_docs) atomicMin(err, p << 1);
      else if (p > term_off[lo] && d <= doc_ids[p - 1]) atomicMin(err, (p << 1) | 1ull);
    }
  }
}

__global__ void sum_u32_kernel(const uint32_t *v, u64 n, u64 *out) {
  u64 s = 0;
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) s += v[i];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, o);
  if ((threadIdx.x & 31) == 0 && s) atomicAdd(out, s);
}

__global__ void df_from_offsets_kernel(const u64 *term_off, uint32_t n_terms, uint32_t *df) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n_terms) df[t] = (uint32_t)(term_off[t + 1] - term_off[t]);
}

// ---- synthetic corpus (SPEC §9), bit-identical to oracle/oracle.c ------------------------------
__constant__ uint16_t c_len_table[OI_LEN_TABLE_SIZE] = OI_LEN_TABLE_INIT;

__global__ void synth_doc_len_kernel(uint64_t seed, uint64_t first_doc, uint64_t n_docs, uint32_t *doc_len) {
  const uint64_t base = oi_stream_base(seed, 2);
  for (u64 d = (u64)blockIdx.x * blockDim.x + threadIdx.x; d < n_docs; d += (u64)gridDim.x * blockDim.x)
    doc_len[d] = c_len_table[oi_cell(oi_row_key(base, first_doc + d), 0) & (OI_LEN_TABLE_SIZE - 1)];
}

__device__ __forceinline__ uint32_t zipf_draw(uint64_t h, const double *__restrict__ cdf, uint32_t vocab) {
  const double u = (double)(h >> 11) * (1.0 / 9007199254740992.0);
  uint32_t lo = 0, hi = vocab - 1;
  while (lo < hi) {
    const uint32_t mid = lo + (hi - lo) / 2;
    if (__ldg(cdf + mid) > u) hi = mid; else lo = mid + 1;
  }
  return lo;
}

// One warp per document: draw the tokens, find the distinct terms and their multiplicities, append
// (term << 32 | local doc, tf) pairs to a global array (order is fixed afterwards by a radix sort).
__global__ void __launch_bounds__(256) synth_postings_kernel(uint64_t seed, uint64_t first_doc, uint64_t n_docs,
                                                             const uint32_t *doc_len, const double *cdf, uint32_t vocab,
                                                             u64 *keys, uint32_t *vals, u64 *n_out) {
  __shared__ uint32_t s_tok[8][256];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint64_t base = oi_stream_base(seed, 3);
  for (u64 d = (u64)blockIdx.x * 8 + warp; d < n_docs; d += (u64)gridDim.x * 8) {
    const uint32_t len = doc_len[d];
    const uint64_t rk = oi_row_key(base, first_doc + d);
    uint32_t *tok = s_tok[warp];
    for (uint32_t i = lane; i < len; i += 32) tok[i] = zipf_draw(oi_cell(rk, i), cdf, vocab);
    __syncwarp();
    for (uint32_t i0 = 0; i0 < len; i0 += 32) {
      const uint32_t i = i0 + lane;
      bool first = false;
      uint32_t tf = 0, t = 0;
      if (i < len) {
        t = tok[i];
        first = true;
        for (uint32_t j = 0; j < len; ++j) {
          const bool same = tok[j] == t;
          tf += same;
          if (same && j < i) first = false;
        }
      }
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, first);
      u64 at = 0;
      if (lane == 0 && m) at = atomicAdd(n_out, (u64)__popc(m));
      at = __shfl_sync(0xFFFFFFFFu, at, 0);
      if (first) {
        const u64 o = at + __popc(m & ((1u << lane) - 1));
        keys[o] = ((u64)t << 32) | (u64)d;
        vals[o] = tf;
      }
    }
    __syncwarp();
  }
}

// sorted (term, doc) keys -> CSR arrays.  Thread i also closes the offsets of the terms between
// its predecessor's term and its own.
__global__ void csr_from_sorted_kernel(const u64 *keys, u64 n, uint32_t n_terms, u64 *term_off, uint32_t *doc_ids) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i <= n; i += (u64)gridDim.x * blockDim.x) {
    const long long t_cur = i < n ? (long long)(keys[i] >> 32) : (long long)n_terms;
    const long long t_prev = i > 0 ? (long long)(keys[i - 1] >> 32) : -1;
    for (long long t = t_prev + 1; t <= t_cur; ++t) term_off[t] = i;
    if (i < n) doc_ids[i] = (uint32_t)keys[i];
  }
}

}  // namespace

void oi_bm25_free(oi_index *h) {
  cudaFree(h->d_vocab); cudaFree(h->d_vocab_off);
  h->d_vocab = nullptr; h->d_vocab_off = nullptr; h->vocab_bytes = 0;
  OiBm25 *b = h->bm25;
  if (!b) return;
  cudaFree(b->d_term_off); cudaFree(b->d_doc_ids); cudaFree(b->d_tfs); cudaFree(b->d_doc_len); cudaFree(b->d_w);
  cudaFree(b->d_post); cudaFree(b->d_dense); cudaFree(b->d_dense_slot); cudaFree(b->d_dense_max);
  cudaFree(b->d_qterms); cudaFree(b->d_qnt); cudaFree(b->d_gthr); cudaFree(b->d_counter); cudaFree(b->d_lists); cudaFree(b->d_best); cudaFree(b->d_qlock);
  cudaFree(b->d_in_terms); cudaFree(b->d_in_offs);
  delete b;
  h->bm25 = nullptr;
}

// capacity of the per-item list workspace in KEYS: up to 1024 lists per query of a full batch at max_k, at most 32 M
// keys (256 MB), at least two lists per query; a call that would need more lowers its item count
static size_t bm25_lists_cap(const oi_index *h) {
  const size_t per = (size_t)h->desc.max_batch * h->desc.max_k;
  const size_t a = std::min<size_t>(1024 * per, (size_t)32 << 20), b = 2 * per;
  return (a > b ? a : b) + 64 * (size_t)h->desc.max_k;
}

static oi_status bm25_alloc_workspace(oi_index *h, OiBm25 *b) {
  const size_t B = h->desc.max_batch;
  OI_CK(cudaMalloc(&b->d_qterms, B * OI_BM25_MAX_QTERMS * sizeof(uint32_t)));
  OI_CK(cudaMalloc(&b->d_qnt, B * sizeof(uint32_t)));
  OI_CK(cudaMalloc(&b->d_gthr, B * sizeof(u64)));
  OI_CK(cudaMalloc(&b->d_counter, sizeof(uint32_t)));
  b->lists_cap = bm25_lists_cap(h);
  OI_CK(cudaMalloc(&b->d_lists, b->lists_cap * sizeof(u64)));
  OI_CK(cudaMalloc(&b->d_best, B * (size_t)h->desc.max_k * sizeof(u64)));
  OI_CK(cudaMalloc(&b->d_qlock, B * sizeof(uint32_t)));
  OI_CK(cudaMalloc(&b->d_in_terms, B * OI_BM25_MAX_QTERMS * sizeof(uint32_t)));
  OI_CK(cudaMalloc(&b->d_in_offs, (B + 1) * sizeof(uint32_t)));
  return OI_OK;
}

extern "C" oi_status oi_index_load_bm25(oi_index *h, const uint64_t *term_offsets, const uint32_t *doc_ids,
                                        const uint32_t *tfs, const uint32_t *doc_len, uint32_t n_terms) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  if (!term_offsets || !doc_len || n_terms == 0) return h->fail(OI_ERR_INVALID_ARG, "NULL CSR array or n_terms == 0");
  const uint64_t P = term_offsets[n_terms];
  if (P && (!doc_ids || !tfs)) return h->fail(OI_ERR_INVALID_ARG, "NULL postings array");
  if (term_offsets[0] != 0) return h->fail(OI_ERR_INVALID_ARG, "term_offsets[0] must be 0");
  for (uint32_t t = 0; t < n_terms; ++t)
    if (term_offsets[t + 1] < term_offsets[t]) return h->fail(OI_ERR_INVALID_ARG, "term_offsets not monotone at term %u", t);
  OI_CK(cudaSetDevice(h->desc.device));
  oi_bm25_free(h);
  OiBm25 *b = new OiBm25();
  h->bm25 = b;
  b->n_terms = n_terms;
  b->n_postings = P;
  const size_t Pa = P ? P : 1;
  OI_CK(cudaMalloc(&b->d_term_off, ((size_t)n_terms + 1) * sizeof(u64)));
  OI_CK(cudaMalloc(&b->d_doc_ids, Pa * sizeof(uint32_t)));
  OI_CK(cudaMalloc(&b->d_tfs, Pa * sizeof(uint32_t)));
  OI_CK(cudaMalloc(&b->d_w, Pa * sizeof(float)));
  OI_CK(cudaMalloc(&b->d_doc_len, (h->desc.n_docs ? h->desc.n_docs : 1) * sizeof(uint32_t)));
  OI_CK(cudaMemcpyAsync(b->d_term_off, term_offsets, ((size_t)n_terms + 1) * sizeof(u64), cudaMemcpyHostToDevice, h->stream));
  if (P) {
    OI_CK(cudaMemcpyAsync(b->d_doc_ids, doc_ids, P * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
    OI_CK(cudaMemcpyAsync(b->d_tfs, tfs, P * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  }
  if (h->desc.n_docs) OI_CK(cudaMemcpyAsync(b->d_doc_len, doc_len, h->desc.n_docs * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
  // the postings are validated where they now are (one pass at HBM speed instead of an O(P) host loop)
  u64 bad = ~0ull;
  if (P) {
    u64 *d_err = nullptr;
    OI_CK(cudaMalloc(&d_err, sizeof(u64)));
    cudaError_t e = cudaMemsetAsync(d_err, 0xFF, sizeof(u64), h->stream);
    if (e == cudaSuccess) {
      bm25_validate_kernel<<<oi_grid(P / 8 + 1, 256, h->num_sms), 256, 0, h->stream>>>(b->d_term_off, b->d_doc_ids, n_terms, P, (uint32_t)h->desc.n_docs, d_err);
      ++h->launches;
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&bad, d_err, sizeof(u64), cudaMemcpyDeviceToHost, h->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
    cudaFree(d_err);
    OI_CK(e);
  } else {
    OI_CK(cudaStreamSynchronize(h->stream));
  }
  if (bad != ~0ull) {
    const uint64_t pb = bad >> 1;
    oi_bm25_free(h);
    if (bad & 1ull) return h->fail(OI_ERR_INVALID_ARG, "posting %llu: doc ids must be strictly ascending inside a list", (unsigned long long)pb);
    return h->fail(OI_ERR_INVALID_ARG, "posting %llu: doc id %u outside the shard", (unsigned long long)pb, doc_ids[pb]);
  }
  return bm25_alloc_workspace(h, b);
}

oi_status oi_bm25_adopt(oi_index *h, uint32_t n_terms, uint64_t n_postings, u64 *d_term_off, uint32_t *d_doc_ids,
                        uint32_t *d_tfs, uint32_t *d_doc_len) {
  oi_bm25_free(h);
  OiBm25 *b = new OiBm25();
  h->bm25 = b;
  b->n_terms = n_terms;
  b->n_postings = n_postings;
  b->d_term_off = d_term_off;
  b->d_doc_ids = d_doc_ids;
  b->d_tfs = d_tfs;
  b->d_doc_len = d_doc_len;
  oi_status s = OI_OK;
  const cudaError_t e = cudaMalloc(&b->d_w, (n_postings ? n_postings : 1) * sizeof(float));
  if (e != cudaSuccess)
    s = h->fail(e == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, "cudaMalloc(weights) failed: %s", cudaGetErrorString(e));
  if (s == OI_OK) s = bm25_alloc_workspace(h, b);
  if (s != OI_OK) oi_bm25_free(h);
  return s;
}

const u64 *oi_bm25_term_offsets(const oi_index *h) { return h->bm25 ? h->bm25->d_term_off : nullptr; }
uint64_t oi_bm25_n_postings(const oi_index *h) { return h->bm25 ? h->bm25->n_postings : 0; }
const uint32_t *oi_bm25_doc_ids(const oi_index *h) { return h->bm25 ? h->bm25->d_doc_ids : nullptr; }
bool oi_bm25_finalized(const oi_index *h) { return h->bm25 && h->bm25->finalized; }

void oi_bm25_replace_terms(oi_index *h, uint32_t n_terms, u64 *d_term_off) {
  OiBm25 *b = h->bm25;
  cudaFree(b->d_term_off);
  b->d_term_off = d_term_off;
  b->n_terms = n_terms;
}

extern "C" oi_status oi_index_synth_bm25(oi_index *h, uint64_t seed, uint32_t vocab, const double *zipf_cdf) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  if (!zipf_cdf || vocab == 0) return h->fail(OI_ERR_INVALID_ARG, "zipf_cdf is NULL or vocab == 0");
  OI_CK(cudaSetDevice(h->desc.device));
  oi_bm25_free(h);
  OiBm25 *b = new OiBm25();
  h->bm25 = b;
  b->n_terms = vocab;
  const u64 n = h->desc.n_docs;
  cudaStream_t st = h->stream;
  double *d_cdf = nullptr;
  u64 *d_cnt = nullptr, *d_keys = nullptr, *d_keys2 = nullptr;
  uint32_t *d_vals = nullptr, *d_vals2 = nullptr;
  void *d_tmp = nullptr;
  auto cleanup = [&]() { cudaFree(d_cdf); cudaFree(d_cnt); cudaFree(d_keys); cudaFree(d_keys2); cudaFree(d_vals); cudaFree(d_vals2); cudaFree(d_tmp); };
#define SY_CK(call)                                                                                       \
  do {                                                                                                    \
    cudaError_t e_ = (call);                                                                              \
    if (e_ != cudaSuccess) {                                                                              \
      cleanup();                                                                                          \
      return h->fail(e_ == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e_)); \
    }                                                                                                     \
  } while (0)
  SY_CK(cudaMalloc(&d_cdf, (size_t)vocab * sizeof(double)));
  SY_CK(cudaMemcpyAsync(d_cdf, zipf_cdf, (size_t)vocab * sizeof(double), cudaMemcpyHostToDevice, st));
  SY_CK(cudaMalloc(&b->d_doc_len, (n ? n : 1) * sizeof(uint32_t)));
  SY_CK(cudaMalloc(&d_cnt, 2 * sizeof(u64)));
  SY_CK(cudaMemsetAsync(d_cnt, 0, 2 * sizeof(u64), st));
  u64 h_cnt[2] = {0, 0};
  if (n) {
    synth_doc_len_kernel<<<oi_grid(n, 256, h->num_sms), 256, 0, st>>>(seed, h->desc.doc_base, n, b->d_doc_len);
    sum_u32_kernel<<<oi_grid(n, 256, h->num_sms), 256, 0, st>>>(b->d_doc_len, n, d_cnt);
    h->launches += 2;
    SY_CK(cudaGetLastError());
    SY_CK(cudaMemcpyAsync(h_cnt, d_cnt, sizeof(u64), cudaMemcpyDeviceToHost, st));
    SY_CK(cudaStreamSynchronize(st));
  }
  const u64 n_tokens = h_cnt[0];
  const size_t cap = n_tokens ? n_tokens : 1;
  SY_CK(cudaMalloc(&d_keys, cap * sizeof(u64)));
  SY_CK(cudaMalloc(&d_vals, cap * sizeof(uint32_t)));
  if (n) {
    u64 blocks = (n + 7) / 8;
    if (blocks > (u64)h->num_sms * 32) blocks = (u64)h->num_sms * 32;
    synth_postings_kernel<<<(unsigned)blocks, 256, 0, st>>>(seed, h->desc.doc_base, n, b->d_doc_len, d_cdf, vocab, d_keys, d_vals, d_cnt + 1);
    ++h->launches;
    SY_CK(cudaGetLastError());
    SY_CK(cudaMemcpyAsync(h_cnt, d_cnt, 2 * sizeof(u64), cudaMemcpyDeviceToHost, st));
    SY_CK(cudaStreamSynchronize(st));
  }
  const u64 P = h_cnt[1];
  b->n_postings = P;
  const size_t Pa = P ? P : 1;
  SY_CK(cudaMalloc(&d_keys2, Pa * sizeof(u64)));
  SY_CK(cudaMalloc(&d_vals2, Pa * sizeof(uint32_t)));
  int term_bits = 1;
  while ((1ull << term_bits) < vocab) ++term_bits;
  const u64 *sorted_keys = d_keys;
  const uint32_t *sorted_vals = d_vals;
  if (P) {
    cub::DoubleBuffer<u64> kb(d_keys, d_keys2);
    cub::DoubleBuffer<uint32_t> vb(d_vals, d_vals2);
    size_t tmp_bytes = 0;
    SY_CK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, kb, vb, P, 0, 32 + term_bits, st));
    SY_CK(cudaMalloc(&d_tmp, tmp_bytes ? tmp_bytes : 1));
    SY_CK(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, kb, vb, P, 0, 32 + term_bits, st));
    h->launches += 8;
    sorted_keys = kb.Current();
    sorted_vals = vb.Current();
  }
  SY_CK(cudaMalloc(&b->d_term_off, ((size_t)vocab + 1) * sizeof(u64)));
  SY_CK(cudaMalloc(&b->d_doc_ids, Pa * sizeof(uint32_t)));
  SY_CK(cudaMalloc(&b->d_tfs, Pa * sizeof(uint32_t)));
  SY_CK(cudaMalloc(&b->d_w, Pa * sizeof(float)));
  csr_from_sorted_kernel<<<oi_grid(P + 1, 256, h->num_sms), 256, 0, st>>>(sorted_keys, P, vocab, b->d_term_off, b->d_doc_ids);
  ++h->launches;
  SY_CK(cudaGetLastError());
  if (P) SY_CK(cudaMemcpyAsync(b->d_tfs, sorted_vals, P * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
  SY_CK(cudaStreamSynchronize(st));
  cleanup();
#undef SY_CK
  return bm25_alloc_workspace(h, b);
}

extern "C" oi_status oi_index_bm25_local_stats(oi_index *h, uint32_t *df_out, uint64_t *sum_doc_len, uint64_t *n_postings) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OiBm25 *b = h->bm25;
  if (!b) return h->fail(OI_ERR_STATE, "no BM25 index loaded");
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  if (n_postings) *n_postings = b->n_postings;
  if (df_out) {
    uint32_t *d_df = nullptr;
    OI_CK(cudaMalloc(&d_df, (size_t)b->n_terms * sizeof(uint32_t)));
    df_from_offsets_kernel<<<(b->n_terms + 255) / 256, 256, 0, st>>>(b->d_term_off, b->n_terms, d_df);
    ++h->launches;
    cudaError_t e = cudaMemcpyAsync(df_out, d_df, (size_t)b->n_terms * sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_df);
    OI_CK(e);
  }
  if (sum_doc_len) {
    u64 *d_s = nullptr;
    OI_CK(cudaMalloc(&d_s, sizeof(u64)));
    cudaError_t e = cudaMemsetAsync(d_s, 0, sizeof(u64), st);
    if (e == cudaSuccess && h->desc.n_docs) {
      sum_u32_kernel<<<oi_grid(h->desc.n_docs, 256, h->num_sms), 256, 0, st>>>(b->d_doc_len, h->desc.n_docs, d_s);
      ++h->launches;
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(sum_doc_len, d_s, sizeof(u64), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_s);
    OI_CK(e);
  }
  return OI_OK;
}

extern "C" oi_status oi_index_bm25_finalize(oi_index *h, const oi_bm25_params *params) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OiBm25 *b = h->bm25;
  if (!b) return h->fail(OI_ERR_STATE, "no BM25 index loaded");
  if (!params || params->struct_size != sizeof(oi_bm25_params)) return h->fail(OI_ERR_INVALID_ARG, "bad oi_bm25_params (struct_size mismatch)");
  if (!(params->k1 >= 0.0f) || !(params->b >= 0.0f && params->b <= 1.0f)) return h->fail(OI_ERR_INVALID_ARG, "k1 must be >= 0 and b in [0, 1]");
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  // df: global if given, else this shard's list lengths
  std::vector<uint32_t> df(b->n_terms);
  // one copy of the offsets (8 B per term) serves both the local df and the choice of the dense columns; the O(P)
  // work -- weights, interleaved postings, dense columns, column maxima -- stays on the device
  std::vector<u64> off((size_t)b->n_terms + 1);
  OI_CK(cudaMemcpyAsync(off.data(), b->d_term_off, off.size() * sizeof(u64), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaStreamSynchronize(st));
  if (params->global_df) {
    std::copy(params->global_df, params->global_df + b->n_terms, df.begin());
  } else {
    for (uint32_t t = 0; t < b->n_terms; ++t) df[t] = (uint32_t)(off[t + 1] - off[t]);
  }
  const uint64_t N = params->n_docs_global ? params->n_docs_global : h->desc.n_docs;
  float avgdl = params->avgdl;
  if (!(avgdl > 0.0f)) {
    u64 *d_s = nullptr, sum = 0;
    OI_CK(cudaMalloc(&d_s, sizeof(u64)));
    cudaError_t e = cudaMemsetAsync(d_s, 0, sizeof(u64), st);
    if (e == cudaSuccess && h->desc.n_docs) {
      sum_u32_kernel<<<oi_grid(h->desc.n_docs, 256, h->num_sms), 256, 0, st>>>(b->d_doc_len, h->desc.n_docs, d_s);
      ++h->launches;
      e = cudaGetLastError();
    }
    if (e == cudaSuccess) e = cudaMemcpyAsync(&sum, d_s, sizeof(u64), cudaMemcpyDeviceToHost, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    cudaFree(d_s);
    OI_CK(e);
    avgdl = h->desc.n_docs ? (float)((double)sum / (double)h->desc.n_docs) : 1.0f;
  }
  // idf: double on the host, rounded once (SPEC §3)
  std::vector<float> idf(b->n_terms);
  for (uint32_t t = 0; t < b->n_terms; ++t) {
    const double d = (double)df[t];
    idf[t] = df[t] == 0 ? 0.0f : (float)std::log(1.0 + ((double)N - d + 0.5) / (d + 0.5));
  }
  // dense columns: the terms present in at least 1/16 of this shard's documents (at most 32, densest first).  At that
  // density a 1024-document block holds >= 64 postings of the term -- a whole chunk -- so streaming the 4-byte column
  // costs no more instructions than walking the 8-byte postings and exposes one load latency instead of several.
  std::vector<int> slot(b->n_terms, -1);
  {
    std::vector<std::pair<u64, uint32_t>> heavy;
    const u64 div = h->bm25_dense_div > 0 ? (u64)h->bm25_dense_div : 16;
    const u64 min_df = std::max<u64>((u64)h->desc.n_docs / div, 1024);
    for (uint32_t t = 0; t < b->n_terms; ++t)
      if (off[t + 1] - off[t] >= min_df) heavy.push_back({off[t + 1] - off[t], t});
    std::sort(heavy.begin(), heavy.end(), [](const std::pair<u64, uint32_t> &x, const std::pair<u64, uint32_t> &y) { return x.first > y.first; });
    if (heavy.size() > OI_BM25_MAX_DENSE) heavy.resize(OI_BM25_MAX_DENSE);
    if (h->bm25_variant == 100) heavy.clear();  // tuning / tests: no dense columns
    for (size_t i = 0; i < heavy.size(); ++i) slot[heavy[i].second] = (int)i;
    b->n_dense = (uint32_t)heavy.size();
  }
  b->dense_stride = (uint32_t)(((size_t)h->desc.n_docs + OI_BM25_ACC_FLOATS - 1) / OI_BM25_ACC_FLOATS * OI_BM25_ACC_FLOATS);
  cudaFree(b->d_post); cudaFree(b->d_dense); cudaFree(b->d_dense_slot); cudaFree(b->d_dense_max);
  b->d_post = nullptr; b->d_dense = nullptr; b->d_dense_slot = nullptr; b->d_dense_max = nullptr;
  const size_t dense_elems = (size_t)std::max<uint32_t>(b->n_dense, 1) * b->dense_stride;
  OI_CK(cudaMalloc(&b->d_post, ((size_t)b->n_postings + OI_BM25_POST_PAD) * sizeof(uint2)));
  OI_CK(cudaMalloc(&b->d_dense, std::max<size_t>(dense_elems, 4) * sizeof(float)));
  OI_CK(cudaMalloc(&b->d_dense_slot, (size_t)b->n_terms * sizeof(int)));
  OI_CK(cudaMemsetAsync(b->d_post, 0xFF, ((size_t)b->n_postings + OI_BM25_POST_PAD) * sizeof(uint2), st));
  OI_CK(cudaMemsetAsync(b->d_dense, 0, std::max<size_t>(dense_elems, 4) * sizeof(float), st));
  OI_CK(cudaMemcpyAsync(b->d_dense_slot, slot.data(), slot.size() * sizeof(int), cudaMemcpyHostToDevice, st));
  OI_CK(cudaMalloc(&b->d_dense_max, OI_BM25_MAX_DENSE * sizeof(float)));
  OI_CK(cudaMemsetAsync(b->d_dense_max, 0, OI_BM25_MAX_DENSE * sizeof(float), st));
  float *d_idf = nullptr;
  OI_CK(cudaMalloc(&d_idf, (size_t)b->n_terms * sizeof(float)));
  cudaError_t e = cudaMemcpyAsync(d_idf, idf.data(), idf.size() * sizeof(float), cudaMemcpyHostToDevice, st);
  if (e == cudaSuccess && b->n_postings) {
    bm25_weights_kernel<<<oi_grid(b->n_postings, 256, h->num_sms), 256, 0, st>>>(b->d_term_off, b->d_doc_ids, b->d_tfs, b->d_doc_len, d_idf,
                                                                                  b->n_terms, b->n_postings, params->k1, params->b, avgdl, b->d_w,
                                                                                  b->d_post, b->d_dense_slot, b->d_dense, b->dense_stride);
    ++h->launches;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess && b->n_dense && h->desc.n_docs) {
    bm25_dense_max_kernel<<<dim3(64, b->n_dense), 256, 0, st>>>(b->d_dense, b->dense_stride, (uint32_t)h->desc.n_docs,
                                                                reinterpret_cast<uint32_t *>(b->d_dense_max));
    ++h->launches;
    e = cudaGetLastError();
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(st);
  cudaFree(d_idf);
  OI_CK(e);
  b->finalized = true;
  return OI_OK;
}

extern "C" oi_status oi_index_read_bm25(oi_index *h, uint64_t *term_offsets, uint32_t *doc_ids, uint32_t *tfs,
                                        uint32_t *doc_len, float *weights) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  OiBm25 *b = h->bm25;
  if (!b) return h->fail(OI_ERR_STATE, "no BM25 index loaded");
  if (weights && !b->finalized) return h->fail(OI_ERR_STATE, "weights requested before oi_index_bm25_finalize");
  OI_CK(cudaSetDevice(h->desc.device));
  cudaStream_t st = h->stream;
  const size_t P = b->n_postings;
  if (term_offsets) OI_CK(cudaMemcpyAsync(term_offsets, b->d_term_off, ((size_t)b->n_terms + 1) * sizeof(u64), cudaMemcpyDeviceToHost, st));
  if (doc_ids && P) OI_CK(cudaMemcpyAsync(doc_ids, b->d_doc_ids, P * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  if (tfs && P) OI_CK(cudaMemcpyAsync(tfs, b->d_tfs, P * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  if (doc_len && h->desc.n_docs) OI_CK(cudaMemcpyAsync(doc_len, b->d_doc_len, h->desc.n_docs * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  if (weights && P) OI_CK(cudaMemcpyAsync(weights, b->d_w, P * sizeof(float), cudaMemcpyDeviceToHost, st));
  OI_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

uint32_t oi_bm25_n_terms(const oi_index *h) { return h->bm25 ? h->bm25->n_terms : 0; }
uint32_t *oi_bm25_stage_terms(oi_index *h) { return h->bm25 ? h->bm25->d_in_terms : nullptr; }
uint32_t *oi_bm25_stage_offs(oi_index *h) { return h->bm25 ? h->bm25->d_in_offs : nullptr; }
size_t oi_bm25_stage_capacity(const oi_index *h) { return (size_t)h->desc.max_batch * OI_BM25_MAX_QTERMS; }

// Enqueues: prep -> blocked scoring -> per-query merge of the S lists into d_out_keys [nq][k]
// (shard-local result, keys carry global doc ids).
oi_status oi_bm25_local_keys(oi_index *h, const uint32_t *d_q_terms, const uint32_t *d_q_offs, uint32_t nq,
                             uint32_t k, u64 *d_out_keys, cudaStream_t st, int overlap) {
  OiBm25 *b = h->bm25;
  if (!b || !b->finalized) return h->fail(OI_ERR_STATE, "BM25 index not loaded / not finalized");
  if (nq == 0) return OI_OK;
  bm25_prep_queries_kernel<<<(nq + 3) / 4, 128, 0, st>>>(d_q_terms, d_q_offs, nq, b->d_term_off, b->n_terms,
                                                             b->d_qterms, b->d_qnt, b->d_gthr, b->d_counter, b->d_best, k, b->d_qlock);
  ++h->launches;
  OI_CK(cudaGetLastError());

  Bm25Params p;
  p.term_off = b->d_term_off; p.doc_ids = b->d_doc_ids; p.post = b->d_post;
  p.dense = b->d_dense; p.dense_slot = b->d_dense_slot; p.dense_max = b->d_dense_max; p.dense_stride = b->dense_stride;
  p.qterms = b->d_qterms; p.qnt = b->d_qnt; p.gthr = b->d_gthr; p.counter = b->d_counter; p.lists = b->d_lists; p.best = b->d_best; p.qlock = b->d_qlock;
  p.n_docs = (uint32_t)h->desc.n_docs; p.doc_base = (uint32_t)h->desc.doc_base; p.nq = nq; p.k = k;
  uint32_t cap = 256;
  while (cap < 2 * k) cap <<= 1;
  p.cap = cap;
  // one warp per work item.  k <= 128: 20 warps per CTA with 2048-document blocks and 2 staged chunks per warp
  // (220 KB of shared memory; 16 warps with 8 chunks each measure 6 % slower); larger k: 8 / 4 / 2 warps with 4096 / 8192 / 16384-document blocks, as many as 64 KB
  // of candidate buffers allow.
  // Tuning options (oi_index_set_option): bm25_warps, bm25_block_docs, bm25_stage_slots; bm25_variant 1..15 keeps
  // its old meaning (warps per CTA rounded down to a power of two, 32768 / warps documents per block).
  const size_t smem_max = 227 * 1024;
  auto smem_for = [&](uint32_t ng_, uint32_t R_, uint32_t ns_) {
    return sizeof(float) * (size_t)ng_ * R_ + (size_t)ng_ * cap * sizeof(u64) + (size_t)ng_ * ns_ * 512 +
           (size_t)ng_ * (sizeof(GrpCtl) + sizeof(u64));
  };
  uint32_t ng = 16;
  while (ng > 1 && ng * cap > 8192) ng >>= 1;
  p.R = OI_BM25_ACC_FLOATS / ng;
  if (cap <= 256) ng = 20;  // 2048-document blocks: 20 x (8 KB scores + 2 KB candidates + 1 KB staging) = 220 KB
  if (h->bm25_variant >= 1 && h->bm25_variant <= 15) {
    uint32_t f = 1;
    while (f * 2 <= (uint32_t)h->bm25_variant) f <<= 1;
    if (f * cap <= 8192) { ng = f; p.R = OI_BM25_ACC_FLOATS / ng; }
  }
  if (h->bm25_warps > 0) ng = (uint32_t)h->bm25_warps;
  if (h->bm25_block_docs > 0) p.R = (uint32_t)h->bm25_block_docs;
  // hybrid overlap mode 1: a CTA small enough (warps x 128 registers, ~106 KB) to share its SM with a GEMM CTA
  const bool lite = overlap == 1 && cap <= 256;
  if (lite) { ng = (uint32_t)h->overlap_bm25_warps; p.R = 2048; }
  if (ng > 24 || p.R < 1024 || (p.R & (p.R - 1)) || smem_for(ng, p.R, 0) > smem_max)
    return h->fail(OI_ERR_INVALID_ARG, "BM25 tuning: %u warps x %u-document blocks (k = %u) do not fit one SM", ng, p.R, k);
  uint32_t nslot = h->bm25_stage_slots >= 0 ? (uint32_t)h->bm25_stage_slots : 8;
  if (lite) nslot = (uint32_t)h->overlap_bm25_slots;
  while (nslot > 0 && smem_for(ng, p.R, nslot) > smem_max) --nslot;
  p.nslot = nslot;
  p.cold_bound = (k <= 256 && nslot >= 2 && !h->bm25_no_cold_bound) ? 1u : 0u;
  p.ng = ng;
  p.r_shift = 0;
  while ((1u << p.r_shift) < p.R) ++p.r_shift;
  p.n_blocks = (p.n_docs + p.R - 1) / p.R;
  if (p.n_blocks == 0) p.n_blocks = 1;
  // one CTA per SM (overlap mode 2: only on the SMs the GEMM leaves free)
  uint32_t grid = (uint32_t)h->num_sms;
  if (overlap == 2) grid = (uint32_t)std::max(1, h->num_sms - h->overlap_gemm_sms);
  const uint32_t groups = grid * ng;
  // super-ranges per query: enough work items (S x nq) for every warp to take ~16, so that the last items to finish
  // (queries differ a lot in cost: zero to several dense terms) leave the SMs idle for a small part of the launch,
  // and items of at most ~32 blocks: the warps in flight then walk a narrow window of the shard (dense columns and
  // postings are re-read from L2, not HBM) and a finished item tightens the query's threshold early.  An item pays a
  // fixed price (one binary search per term, one fold), which is what keeps items from being smaller still
  // (sweeps at 6.25M / 12.5M / 50M documents, batch 256, and 10M, batch 1024: docs/NOTES_r02.md).
  uint32_t ipw = h->bm25_items_per_warp > 0 ? (uint32_t)h->bm25_items_per_warp : 16;
  uint32_t S = (ipw * groups + nq - 1) / nq;
  if (h->bm25_items_per_warp <= 0) S = std::max(std::min(S, 256u), (p.n_blocks + 31) / 32);
  if (S < 1) S = 1;
  if (S > 1024) S = 1024;  // the per-query merge is one CTA per query: its prefix tables hold 1024 lists
  while (S > 1 && (size_t)S * nq * k > b->lists_cap) --S;
  if (S > p.n_blocks) S = p.n_blocks;
  p.J = (p.n_blocks + S - 1) / S;
  p.S = (p.n_blocks + p.J - 1) / p.J;
  if ((size_t)p.S * nq * k > b->lists_cap) return h->fail(OI_ERR_CUDA, "internal: BM25 list workspace too small (%u x %u)", p.S, nq);
  const size_t smem = smem_for(ng, p.R, nslot);
  if (!b->attr_set) {  // once per index (the attribute is per function and device)
    OI_CK(cudaFuncSetAttribute(bm25_blocked_kernel<512, 2048>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    OI_CK(cudaFuncSetAttribute(bm25_blocked_kernel<512, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    OI_CK(cudaFuncSetAttribute(bm25_blocked_kernel<768, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    OI_CK(cudaFuncSetAttribute(bm25_blocked_kernel<576, 2048>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    OI_CK(cudaFuncSetAttribute(bm25_blocked_kernel<640, 2048>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    b->attr_set = true;
  }
  // one CTA per SM; with fewer items than SMs x warps the items still spread over all SMs (each SM's first warps
  // to reach the counter take them): a single query is latency-bound and every SM brings its own load pipes
  if (grid > p.S * nq) grid = p.S * nq;
  if (ng > 16 && ng <= 18 && p.R == 2048) bm25_blocked_kernel<576, 2048><<<grid, ng * 32, smem, st>>>(p);
  else if (ng > 18 && ng <= 20 && p.R == 2048) bm25_blocked_kernel<640, 2048><<<grid, ng * 32, smem, st>>>(p);
  else if (ng > 16) bm25_blocked_kernel<768, 0><<<grid, ng * 32, smem, st>>>(p);
  else if (p.R == 2048) bm25_blocked_kernel<512, 2048><<<grid, ng * 32, smem, st>>>(p);
  else bm25_blocked_kernel<512, 0><<<grid, ng * 32, smem, st>>>(p);
  ++h->launches;
  OI_CK(cudaGetLastError());
#ifdef OI_BM25_STATS
  bm25_stats_print_kernel<<<1, 1, 0, st>>>();
#endif
  OI_CK(oi_launch_merge_shards(b->d_lists, p.S, nq, k, d_out_keys, st, &h->launches, 0, b->d_gthr));
  return OI_OK;
}
