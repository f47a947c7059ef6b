// lexicon.cu — batched GPU PostAnalyzer: the reference's LexiconAnalyzer::score
// (src/adapters/analyzer/lexicon.rs:53-73, word lists :9-44) over a whole batch of posts.
//
// Tokenizer (lexicon.rs:54-58; docs/SPEC.md §6): Unicode-lowercase, split on every char that is
// not ASCII alphanumeric.  On UTF-8 bytes: ASCII letters/digits are token bytes (A-Z lowered),
// every other byte is a separator, except U+212A KELVIN SIGN (E2 84 AA -> 'k', its two
// continuation bytes are transparent) and U+0130 (C4 B0 -> 'i' followed by a separator).
//
// One warp per post; lanes stride over the byte positions.  A lane that sits on the first byte of
// a token gathers its (<= 9 relevant) normalised bytes into a 128-bit word and compares it with
// the packed BULL / BEAR / JARGON tables.  Integer hit counts are exact; polarity is one f64
// divide (Polarity::new clamps to [-1, 1], src/domain/values/polarity.rs:8-14).
// The post is staged once into shared memory (coalesced 16-byte loads; posts longer than the staging area are read in
// place), so the tokenizer's look-back / look-ahead reads never go back to global memory: algorithmic bytes = the text
// bytes, read once.  The kernel is instruction-bound, not HBM-bound (~25 instructions per byte); see
// profiles/r02_ncu_lexicon.md.
//
// Handle-based API (round 2): oi_lexicon_create allocates the stream and the device buffers once; oi_lexicon_run reuses
// them (they grow on demand) and can fuse the reference's social summary (SpeculationEngine::social_summary,
// src/domain/engine/speculation_engine.rs:70-125) into the same call.  oi_lexicon_analyze keeps its round-1 signature
// on top of a per-device cached handle.
#include <map>
#include <mutex>
#include <string>

#include "internal.h"
#include "oi_summary.cuh"
#include "oi_tokenize.cuh"

namespace {

struct Word { unsigned long long lo, hi; };

constexpr Word pack_word(const char *s) {
  unsigned long long lo = 0, hi = 0;
  int i = 0;
  for (; s[i] && i < 8; ++i) lo |= (unsigned long long)(unsigned char)s[i] << (8 * i);
  for (; s[i] && i < 16; ++i) hi |= (unsigned long long)(unsigned char)s[i] << (8 * (i - 8));
  return Word{lo, hi};
}

constexpr int N_BULL = 14, N_BEAR = 13, N_JARGON = 15;
__constant__ Word c_bull[N_BULL] = {pack_word("moon"), pack_word("calls"), pack_word("long"), pack_word("buy"),
                                    pack_word("bullish"), pack_word("squeeze"), pack_word("breakout"),
                                    pack_word("rocket"), pack_word("pump"), pack_word("rip"), pack_word("green"),
                                    pack_word("up"), pack_word("rally"), pack_word("bull")};
__constant__ Word c_bear[N_BEAR] = {pack_word("puts"), pack_word("short"), pack_word("sell"), pack_word("bearish"),
                                    pack_word("dump"), pack_word("crash"), pack_word("drilling"),
                                    pack_word("bagholder"), pack_word("rug"), pack_word("red"), pack_word("down"),
                                    pack_word("tank"), pack_word("bear")};
__constant__ Word c_jargon[N_JARGON] = {pack_word("calls"), pack_word("puts"), pack_word("0dte"), pack_word("yolo"),
                                        pack_word("leaps"), pack_word("theta"), pack_word("gamma"),
                                        pack_word("squeeze"), pack_word("otm"), pack_word("itm"), pack_word("strike"),
                                        pack_word("iv"), pack_word("delta"), pack_word("vega"), pack_word("contracts")};

// The 39 distinct list words in a 128-slot perfect hash (the multiplier was searched offline: no two words share a slot),
// built in shared memory at kernel start from the tables above: a token costs one multiply, one table read and one
// 128-bit compare instead of 42 compares (ncu, round 1 layout: 9.2 G warp instructions for 300 MB of text).
struct LexSlot { unsigned long long lo, hi; uint32_t flags, pad; };  // flags: 1 = BULL, 2 = BEAR, 4 = JARGON
constexpr int kLexSlots = 128;
__host__ __device__ __forceinline__ uint32_t lex_hash(unsigned long long lo, unsigned long long hi) {
  return (uint32_t)(((lo ^ (hi * 0x9E3779B97F4A7C15ull)) * 0x3CDFA3C5131A5AF7ull) >> 57);
}

constexpr int kStageBytes = 4096;  // per warp: posts up to this many bytes are tokenized from shared memory

__global__ void __launch_bounds__(256) lexicon_kernel(const uint8_t *texts, const unsigned long long *offsets,
                                                      unsigned long long n_posts, double *polarity,
                                                      uint8_t *speculative, uint32_t *bull_hits, uint32_t *bear_hits) {
  __shared__ __align__(16) uint8_t s_stage[8][kStageBytes + 32];
  __shared__ LexSlot s_tab[kLexSlots];
  if (threadIdx.x < kLexSlots) s_tab[threadIdx.x] = LexSlot{0ull, 0ull, 0u, 0u};
  __syncthreads();
  if (threadIdx.x < N_BULL + N_BEAR + N_JARGON) {
    const int w = threadIdx.x;
    const Word wd = w < N_BULL ? c_bull[w] : (w < N_BULL + N_BEAR ? c_bear[w - N_BULL] : c_jargon[w - N_BULL - N_BEAR]);
    LexSlot *e = &s_tab[lex_hash(wd.lo, wd.hi)];
    e->lo = wd.lo;  // a word that is in two lists writes the same key twice
    e->hi = wd.hi;
    atomicOr(&e->flags, w < N_BULL ? 1u : (w < N_BULL + N_BEAR ? 2u : 4u));
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const unsigned long long warp = ((unsigned long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const unsigned long long n_warps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
  uint8_t *stage = s_stage[threadIdx.x >> 5];
  for (unsigned long long post = warp; post < n_posts; post += n_warps) {
    const uint8_t *t = texts + offsets[post];
    const long long len = (long long)(offsets[post + 1] - offsets[post]);
    bool ascii = false;
    if (len <= kStageBytes) {
      // the 16-byte words that cover the post, loaded aligned (the allocation is padded to whole words); the post's
      // first byte sits at `sh` inside the staged copy
      const uintptr_t a0 = reinterpret_cast<uintptr_t>(t) & ~(uintptr_t)15;
      const int sh = (int)(reinterpret_cast<uintptr_t>(t) - a0);
      const int n_words = (int)((sh + len + 15) >> 4);
      __syncwarp();  // the previous post's readers are done with the staging area
      uint32_t hb = 0;
      for (int w = lane; w < n_words; w += 32) {
        const uint4 v = __ldg(reinterpret_cast<const uint4 *>(a0) + w);
        reinterpret_cast<uint4 *>(stage)[w] = v;
        hb |= v.x | v.y | v.z | v.w;
      }
      __syncwarp();
      t = stage + sh;
      // no byte >= 0x80 in the covering words (a neighbour's bytes in the first / last word only make this conservative)
      ascii = !__any_sync(0xFFFFFFFFu, (hb & 0x80808080u) != 0u);
    }
    uint32_t bull = 0, bear = 0, spec = 0;
    if (ascii) {
      // ASCII fast path (the usual post): 32 bytes per step, one ballot finds the token starts, and every start lane
      // reads its token as 16 bytes + 1 from shared memory and classifies / lowercases them four at a time (SWAR) --
      // no per-byte loop.  Same tokens, same packing as the general path below.
      uint32_t carry = 0;  // was the last byte of the previous step a token byte
      for (long long c0 = 0; c0 < len; c0 += 32) {
        const long long i = c0 + lane;
        const uint32_t b = i < len ? (uint32_t)t[i] : 0x20u;
        const bool tok = oi_ascii_token_byte(b);
        const uint32_t m = __ballot_sync(0xFFFFFFFFu, tok);
        const uint32_t starts = m & ~((m << 1) | carry);
        carry = m >> 31;
        if (!((starts >> lane) & 1u)) continue;
        const uintptr_t addr = reinterpret_cast<uintptr_t>(t + i);
        const uint32_t *wp = reinterpret_cast<const uint32_t *>(addr & ~(uintptr_t)3);
        const uint32_t sh8 = (uint32_t)(addr & 3u) * 8u;
        const uint32_t w0 = wp[0], w1 = wp[1], w2 = wp[2], w3 = wp[3], w4 = wp[4];
        uint32_t x[4] = {__funnelshift_r(w0, w1, sh8), __funnelshift_r(w1, w2, sh8), __funnelshift_r(w2, w3, sh8),
                         __funnelshift_r(w3, w4, sh8)};
        const uint32_t b16 = (w4 >> sh8) & 0xFFu;
        uint32_t n = 0;
        bool run = true;  // still inside the token's leading run
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          // bytes are < 0x80: x + (0x80 - lo) sets bit 7 iff x >= lo, no carry into the next byte
          const uint32_t v = x[u];
          const uint32_t up = (v + 0x3F3F3F3Fu) & ~(v + 0x25252525u);  // 'A' .. 'Z'
          const uint32_t lw = (v + 0x1F1F1F1Fu) & ~(v + 0x05050505u);  // 'a' .. 'z'
          const uint32_t dg = (v + 0x50505050u) & ~(v + 0x46464646u);  // '0' .. '9'
          const uint32_t tm = (up | lw | dg) & 0x80808080u;
          x[u] = v | ((up & 0x80808080u) >> 2);                         // lower the capitals
          const uint32_t nt = ~tm & 0x80808080u;
          const uint32_t lead = nt ? (uint32_t)(__ffs((int)nt) - 1) >> 3 : 4u;
          if (run) n += lead;
          run = run && lead == 4u;
        }
        const bool more = run && oi_ascii_token_byte(b16);  // a 17th token byte
        const long long left = len - i;
        if (more && left > 16) continue;  // longer than 16 bytes: cannot match a list word
        if ((long long)n > left) n = (uint32_t)left;
        unsigned long long lo = (unsigned long long)x[0] | ((unsigned long long)x[1] << 32);
        unsigned long long hi = (unsigned long long)x[2] | ((unsigned long long)x[3] << 32);
        if (n < 8) { lo &= (1ull << (8 * n)) - 1ull; hi = 0ull; }
        else if (n < 16) hi &= (1ull << (8 * (n - 8))) - 1ull;
        const LexSlot e = s_tab[lex_hash(lo, hi)];
        const uint32_t f = (e.lo == lo && e.hi == hi) ? e.flags : 0u;
        bull += f & 1u;
        bear += (f >> 1) & 1u;
        spec |= (f >> 2) & 1u;
      }
    } else
    for (long long i = lane; i < len; i += 32) {
      const int c = classify(t, i, len);
      if (c == CLS_SEP || c == CLS_SKIP) continue;
      // token start? look back over transparent bytes to the previous real position
      long long j = i - 1;
      while (j >= 0 && classify(t, j, len) == CLS_SKIP) --j;
      if (j >= 0) {
        const int pc = classify(t, j, len);
        if (pc > 0) continue;  // previous char continues the same token (U+0130's 'i' ends one: pc < 0)
      }
      // gather the token: up to 16 bytes, anything longer cannot match a list word
      unsigned long long lo = 0, hi = 0;
      int n = 0;
      long long p = i;
      int cc = c;
      for (;;) {
        const int ch = cc == CLS_I_THEN_SEP ? 'i' : cc;
        if (n < 8) lo |= (unsigned long long)ch << (8 * n);
        else if (n < 16) hi |= (unsigned long long)ch << (8 * (n - 8));
        ++n;
        if (cc == CLS_I_THEN_SEP || n > 16) break;
        ++p;
        while (p < len && (cc = classify(t, p, len)) == CLS_SKIP) ++p;
        if (p >= len || cc == CLS_SEP) break;
      }
      const bool too_long = n > 16;
      if (too_long) continue;
      const LexSlot e = s_tab[lex_hash(lo, hi)];
      const uint32_t f = (e.lo == lo && e.hi == hi) ? e.flags : 0u;
      bull += f & 1u;
      bear += (f >> 1) & 1u;
      spec |= (f >> 2) & 1u;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      bull += __shfl_xor_sync(0xFFFFFFFFu, bull, o);
      bear += __shfl_xor_sync(0xFFFFFFFFu, bear, o);
      spec |= __shfl_xor_sync(0xFFFFFFFFu, spec, o);
    }
    if (lane == 0) {
      const double bh = (double)bull, eh = (double)bear;
      double pol = (bh + eh == 0.0) ? 0.0 : (bh - eh) / (bh + eh);
      if (pol != pol) pol = 0.0;
      pol = pol > 1.0 ? 1.0 : (pol < -1.0 ? -1.0 : pol);
      polarity[post] = pol;
      speculative[post] = (uint8_t)(spec != 0);
      if (bull_hits) bull_hits[post] = bull;
      if (bear_hits) bear_hits[post] = bear;
    }
  }
}

}  // namespace

void oi_set_thread_error(const std::string &msg);  // api.cu

// The reference's social summary over the batch's signals (src/domain/engine/speculation_engine.rs:76-84): one CTA, the
// shared summary body (oi_summary.cuh) over the identity order.
__global__ void __launch_bounds__(128) social_summary_kernel(const double *polarity, const uint8_t *speculative, unsigned long long n, double thr,
                                                             oi_social_summary *out) {
  oi_social_summary_cta<false>(polarity, speculative, nullptr, 0ull, n, -1, thr, nullptr, nullptr, out);
}

struct oi_lexicon {
  int device = 0;
  cudaStream_t st = nullptr;
  std::mutex mu;
  uint8_t *d_text = nullptr, *d_spec = nullptr;
  unsigned long long *d_off = nullptr;
  double *d_pol = nullptr;
  uint32_t *d_bull = nullptr, *d_bear = nullptr;
  oi_social_summary *d_sum = nullptr;
  size_t cap_bytes = 0, cap_posts = 0;
  uint64_t launches = 0;
};

static oi_status lx_fail(oi_status code, const std::string &m) { oi_set_thread_error(m); return code; }

#define LX_CK(call)                                                                                  \
  do {                                                                                               \
    cudaError_t e_ = (call);                                                                         \
    if (e_ != cudaSuccess)                                                                           \
      return lx_fail(e_ == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA,           \
                     std::string(#call " failed: ") + cudaGetErrorString(e_));                       \
  } while (0)

// (re)allocates the device buffers so that a batch of `bytes` text bytes / `posts` posts fits
static oi_status lx_reserve(oi_lexicon *lx, size_t bytes, size_t posts) {
  if (bytes > lx->cap_bytes) {
    cudaFree(lx->d_text);
    lx->d_text = nullptr;
    lx->cap_bytes = 0;
    const size_t want = bytes + bytes / 4 + 64;  // + two 16-byte words: the staging loads read whole aligned words
    LX_CK(cudaMalloc(&lx->d_text, want + 32));
    lx->cap_bytes = want;
  }
  if (posts > lx->cap_posts) {
    cudaFree(lx->d_off); cudaFree(lx->d_pol); cudaFree(lx->d_spec); cudaFree(lx->d_bull); cudaFree(lx->d_bear);
    lx->d_off = nullptr; lx->d_pol = nullptr; lx->d_spec = nullptr; lx->d_bull = nullptr; lx->d_bear = nullptr;
    lx->cap_posts = 0;
    const size_t want = posts + posts / 4 + 16;
    LX_CK(cudaMalloc(&lx->d_off, (want + 1) * sizeof(unsigned long long)));
    LX_CK(cudaMalloc(&lx->d_pol, want * sizeof(double)));
    LX_CK(cudaMalloc(&lx->d_spec, want));
    LX_CK(cudaMalloc(&lx->d_bull, want * sizeof(uint32_t)));
    LX_CK(cudaMalloc(&lx->d_bear, want * sizeof(uint32_t)));
    lx->cap_posts = want;
  }
  return OI_OK;
}

extern "C" oi_status oi_lexicon_create(int32_t device, uint64_t reserve_bytes, uint64_t reserve_posts, oi_lexicon **out) {
  if (!out) return lx_fail(OI_ERR_INVALID_ARG, "out is NULL");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return lx_fail(OI_ERR_NO_DEVICE, std::string("no CUDA device: ") + cudaGetErrorString(e) + " (this library has no CPU fallback)");
  if (device < 0 || device >= n_dev) return lx_fail(OI_ERR_INVALID_ARG, "device ordinal out of range");
  oi_lexicon *lx = new (std::nothrow) oi_lexicon();
  if (!lx) return lx_fail(OI_ERR_OUT_OF_MEMORY, "host allocation failed");
  lx->device = device;
  oi_status s = OI_OK;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&lx->st, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaMalloc(&lx->d_sum, sizeof(oi_social_summary))) != cudaSuccess)
    s = lx_fail(OI_ERR_CUDA, std::string("lexicon handle: ") + cudaGetErrorString(e));
  if (s == OI_OK) s = lx_reserve(lx, (size_t)reserve_bytes, (size_t)reserve_posts);
  if (s != OI_OK) { oi_lexicon_destroy(lx); return s; }
  *out = lx;
  return OI_OK;
}

extern "C" void oi_lexicon_destroy(oi_lexicon *lx) {
  if (!lx) return;
  cudaSetDevice(lx->device);
  if (lx->st) cudaStreamSynchronize(lx->st);
  cudaFree(lx->d_text); cudaFree(lx->d_off); cudaFree(lx->d_pol); cudaFree(lx->d_spec); cudaFree(lx->d_bull); cudaFree(lx->d_bear);
  cudaFree(lx->d_sum);
  if (lx->st) cudaStreamDestroy(lx->st);
  delete lx;
}

extern "C" oi_status oi_lexicon_run(oi_lexicon *lx, const uint8_t *texts, const uint64_t *offsets, uint64_t n_posts,
                                    double *out_polarity, uint8_t *out_speculative, uint32_t *out_bull_hits,
                                    uint32_t *out_bear_hits, double bull_bear_threshold, oi_social_summary *out_summary) {
  if (!lx) return lx_fail(OI_ERR_INVALID_ARG, "lexicon handle is NULL");
  std::lock_guard<std::mutex> lock(lx->mu);
  if (n_posts == 0) {
    if (out_summary) { *out_summary = oi_social_summary(); out_summary->bull_bear_ratio = -1.0; }
    return OI_OK;
  }
  if (!offsets || !out_polarity || !out_speculative) return lx_fail(OI_ERR_INVALID_ARG, "NULL offsets / output pointer");
  for (uint64_t i = 0; i < n_posts; ++i)
    if (offsets[i + 1] < offsets[i]) return lx_fail(OI_ERR_INVALID_ARG, "offsets not monotone");
  const uint64_t n_bytes = offsets[n_posts] - offsets[0];
  if (n_bytes && !texts) return lx_fail(OI_ERR_INVALID_ARG, "texts is NULL");
  LX_CK(cudaSetDevice(lx->device));
  oi_status s = lx_reserve(lx, (size_t)n_bytes, (size_t)n_posts);
  if (s) return s;
  cudaStream_t st = lx->st;
  // the blob lands 16-byte aligned at d_text + 16, so that the word-wise staging of the first post may read the word below
  uint8_t *d_blob = lx->d_text + 16;
  if (n_bytes) LX_CK(cudaMemcpyAsync(d_blob, texts + offsets[0], n_bytes, cudaMemcpyHostToDevice, st));
  LX_CK(cudaMemcpyAsync(lx->d_off, offsets, (n_posts + 1) * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
  uint64_t blocks = (n_posts + 7) / 8;
  if (blocks > 148ull * 8) blocks = 148ull * 8;
  // offsets are rebased to the copied blob on the device side by passing the blob pointer minus offsets[0]
  lexicon_kernel<<<(unsigned)blocks, 256, 0, st>>>(d_blob - offsets[0], lx->d_off, n_posts, lx->d_pol, lx->d_spec, lx->d_bull, lx->d_bear);
  ++lx->launches;
  LX_CK(cudaGetLastError());
  if (out_summary) {
    social_summary_kernel<<<1, 128, 0, st>>>(lx->d_pol, lx->d_spec, n_posts, bull_bear_threshold, lx->d_sum);
    ++lx->launches;
    LX_CK(cudaGetLastError());
    LX_CK(cudaMemcpyAsync(out_summary, lx->d_sum, sizeof(oi_social_summary), cudaMemcpyDeviceToHost, st));
  }
  LX_CK(cudaMemcpyAsync(out_polarity, lx->d_pol, n_posts * sizeof(double), cudaMemcpyDeviceToHost, st));
  LX_CK(cudaMemcpyAsync(out_speculative, lx->d_spec, n_posts, cudaMemcpyDeviceToHost, st));
  if (out_bull_hits) LX_CK(cudaMemcpyAsync(out_bull_hits, lx->d_bull, n_posts * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  if (out_bear_hits) LX_CK(cudaMemcpyAsync(out_bear_hits, lx->d_bear, n_posts * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  LX_CK(cudaStreamSynchronize(st));
  return OI_OK;
}

extern "C" uint64_t oi_lexicon_launch_count(const oi_lexicon *lx) { return lx ? lx->launches : 0; }

// round-1 entry point: the same call on a per-device handle that is created on first use and kept for the process
extern "C" oi_status oi_lexicon_analyze(int32_t device, const uint8_t *texts, const uint64_t *offsets,
                                        uint64_t n_posts, double *out_polarity, uint8_t *out_speculative,
                                        uint32_t *out_bull_hits, uint32_t *out_bear_hits) {
  static std::mutex mu;
  static std::map<int, oi_lexicon *> cache;
  oi_lexicon *lx = nullptr;
  {
    std::lock_guard<std::mutex> lock(mu);
    auto it = cache.find(device);
    if (it == cache.end()) {
      oi_status s = oi_lexicon_create(device, 1 << 20, 1 << 12, &lx);
      if (s) return s;
      cache[device] = lx;
    } else {
      lx = it->second;
    }
  }
  return oi_lexicon_run(lx, texts, offsets, n_posts, out_polarity, out_speculative, out_bull_hits, out_bear_hits, 0.2, nullptr);
}
#undef LX_CK
