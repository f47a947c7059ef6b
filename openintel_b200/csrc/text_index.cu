// text_index.cu — posts -> this shard's BM25 part, on the device (oi_index_build_bm25_text): tokenizer, vocabulary and
// CSR in one call, bit-identical to the host IndexBuilder (openintel_b200/host/openintel_host.hpp; docs/SPEC.md §3).
//
//   1. count pass, one warp per post: every lane classifies one byte (oi_tokenize.cuh, the lexicon scorer's rules), one
//      ballot finds the token bytes and one the token starts.  -> tokens per post (= doc_len) and token bytes per post.
//   2. two exclusive scans give every post its first occurrence slot and its place in the token-byte arena.
//   3. emit pass, the same walk: each token's lowered bytes go to the arena, each occurrence records (arena offset, doc).
//      Occurrences come out in (doc, position) order.
//   4. key: the token's first 12 bytes in base 37 (end = 0, '0'..'9' = 1..10, 'a'..'z' = 11..36) -- tokens are
//      [0-9a-z] only, so the numeric order of the keys is the byte order of the tokens, and 37^12 < 2^63.
//      One stable radix sort of (key, occurrence).  Tokens of 12 bytes or more can share a key (all of them have a
//      non-zero last digit); those occurrences are re-sorted among themselves by a stable merge sort on the full bytes
//      and written back into the same slots.  Both sorts are stable and the occurrences were in doc order, so every
//      term's occurrences end up grouped and in ascending doc order.
//   5. boundaries: one flag word per sorted occurrence (new term << 32 | new (term, doc)), one inclusive scan -> term
//      ranks, posting slots, term_offsets, doc ids, tf = run lengths, and the vocabulary (one token per term).
//   6. hand-off: the CSR is adopted as the index's BM25 part (oi_bm25_adopt), exactly as oi_index_load_bm25 leaves it.
//
// Step 4 is one helper (RecordSort) that sorts any (arena, offsets) records into byte order; the vocabulary union of a
// document-sharded index (oi_index_bm25_union_vocabulary, below) runs the shards' vocabulary entries through it.
//
// The tokenizer passes read the text in place from global memory (the look-back / look-ahead of classify() hits L1), so
// a post of any length takes the same path.
#include <cub/device/device_merge_sort.cuh>
#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

#include "handle.h"
#include "oi_tokenize.cuh"

namespace {

constexpr int kKeyChars = 12;

// one warp per post.  EMIT = false: tokens and token bytes per post; EMIT = true: arena bytes and occurrences
template <bool EMIT>
__global__ void __launch_bounds__(256) text_tokens_kernel(const uint8_t *texts, const u64 *offsets, u64 n_posts, u64 *n_tok,
                                                          u64 *n_chr, uint32_t *doc_len, uint8_t *arena, u64 *occ_off,
                                                          uint32_t *occ_doc) {
  const int lane = threadIdx.x & 31;
  const uint32_t below = (1u << lane) - 1u;
  const u64 warp = ((u64)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const u64 n_warps = ((u64)gridDim.x * blockDim.x) >> 5;
  for (u64 post = warp; post < n_posts; post += n_warps) {
    const uint8_t *t = texts + offsets[post];
    const long long len = (long long)(offsets[post + 1] - offsets[post]);
    // EMIT: the scanned counts of the count pass = this post's first occurrence slot and first arena byte
    u64 toks = EMIT ? n_tok[post] : 0, chrs = EMIT ? n_chr[post] : 0;
    for (long long c0 = 0; c0 < len; c0 += 32) {
      const long long i = c0 + lane;
      int c = CLS_SEP;
      bool start = false;
      if (i < len) {
        c = classify(t, i, len);
        if (c > 0 || c == CLS_I_THEN_SEP) {
          // a token starts here unless the previous real position (transparent bytes skipped) continues a token;
          // U+0130's 'i' ends its token (class < 0)
          long long j = i - 1;
          while (j >= 0 && classify(t, j, len) == CLS_SKIP) --j;
          start = j < 0 || classify(t, j, len) <= 0;
        }
      }
      const bool chr = c > 0 || c == CLS_I_THEN_SEP;
      const uint32_t cm = __ballot_sync(0xFFFFFFFFu, chr), sm = __ballot_sync(0xFFFFFFFFu, start);
      if (EMIT) {
        const u64 at = chrs + __popc(cm & below);
        if (chr) arena[at] = (uint8_t)(c > 0 ? c : 'i');
        if (start) {
          const u64 o = toks + __popc(sm & below);
          occ_off[o] = at;
          occ_doc[o] = (uint32_t)post;
        }
      }
      chrs += __popc(cm);
      toks += __popc(sm);
    }
    if (!EMIT && lane == 0) {
      n_tok[post] = toks;
      n_chr[post] = chrs;
      doc_len[post] = (uint32_t)toks;
    }
  }
}

// occurrence o = arena[occ_off[o] .. occ_off[o + 1]) -> its 12-byte base-37 key; vals = o
__global__ void text_keys_kernel(const uint8_t *arena, const u64 *occ_off, u64 n, u64 *keys, uint32_t *vals) {
  for (u64 o = (u64)blockIdx.x * blockDim.x + threadIdx.x; o < n; o += (u64)gridDim.x * blockDim.x) {
    const u64 a = occ_off[o], len = occ_off[o + 1] - a;
    u64 k = 0;
#pragma unroll
    for (int i = 0; i < kKeyChars; ++i) {
      uint32_t d = 0;
      if ((u64)i < len) {
        const uint32_t ch = arena[a + i];
        d = ch <= '9' ? ch - '0' + 1 : ch - 'a' + 11;
      }
      k = k * 37 + d;
    }
    keys[o] = k;
    vals[o] = (uint32_t)o;
  }
}

// the key of a token of at least 12 bytes ends in a non-zero digit; only such keys can be shared by different tokens
__host__ __device__ __forceinline__ bool key_may_collide(u64 key) { return key % 37 != 0; }

struct KeyMayCollide {
  const u64 *keys;
  __device__ bool operator()(uint32_t i) const { return key_may_collide(keys[i]); }
};

// byte order of two occurrences' tokens (a proper prefix sorts first)
struct TokenLess {
  const uint8_t *arena;
  const u64 *occ_off;
  __device__ bool operator()(uint32_t a, uint32_t b) const {
    const uint8_t *x = arena + occ_off[a], *y = arena + occ_off[b];
    const u64 la = occ_off[a + 1] - occ_off[a], lb = occ_off[b + 1] - occ_off[b];
    const u64 n = la < lb ? la : lb;
    for (u64 i = 0; i < n; ++i)
      if (x[i] != y[i]) return x[i] < y[i];
    return la < lb;
  }
};

__device__ bool same_token(const uint8_t *arena, const u64 *occ_off, uint32_t a, uint32_t b) {
  const u64 la = occ_off[a + 1] - occ_off[a];
  if (occ_off[b + 1] - occ_off[b] != la) return false;
  const uint8_t *x = arena + occ_off[a], *y = arena + occ_off[b];
  for (u64 i = kKeyChars; i < la; ++i)  // the first 12 bytes are equal: same key
    if (x[i] != y[i]) return false;
  return true;
}

// the key-equality test of the sorted records (RecordSort): record i > 0 in sorted order holds the same bytes as i - 1
__device__ __forceinline__ bool same_as_previous(const u64 *keys, const uint32_t *order, const uint8_t *arena,
                                                 const u64 *off, u64 i) {
  return keys[i] == keys[i - 1] && (!key_may_collide(keys[i]) || same_token(arena, off, order[i - 1], order[i]));
}

__global__ void gather_kernel(const uint32_t *src, const uint32_t *idx, uint32_t n, uint32_t *dst) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) dst[j] = src[idx[j]];
}
__global__ void scatter_kernel(const uint32_t *src, const uint32_t *idx, uint32_t n, uint32_t *dst) {
  for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += gridDim.x * blockDim.x) dst[idx[j]] = src[j];
}

// sorted occurrence i -> (starts a term) << 32 | (starts a posting)
__global__ void text_flags_kernel(const u64 *keys, const uint32_t *occ, const uint8_t *arena, const u64 *occ_off,
                                  const uint32_t *occ_doc, u64 n, u64 *flags) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    bool nt = true, np = true;
    if (i > 0) {
      nt = !same_as_previous(keys, occ, arena, occ_off, i);
      np = nt || occ_doc[occ[i - 1]] != occ_doc[occ[i]];
    }
    flags[i] = ((u64)nt << 32) | (u64)np;
  }
}

// scanned flags -> term_off[n_terms + 1], doc_ids[P], posting starts pstart[P + 1] (in sorted occurrences), the first
// occurrence of every term
__global__ void text_csr_kernel(const u64 *scan, const uint32_t *occ, const uint32_t *occ_doc, u64 n, u64 *term_off,
                                uint32_t *doc_ids, uint32_t *pstart, uint32_t *first_occ) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x) {
    const u64 s = scan[i], prev = i ? scan[i - 1] : 0;
    const uint32_t p = (uint32_t)s - 1u, t = (uint32_t)(s >> 32) - 1u;
    if ((uint32_t)s != (uint32_t)prev) {
      doc_ids[p] = occ_doc[occ[i]];
      pstart[p] = (uint32_t)i;
    }
    if ((s >> 32) != (prev >> 32)) {
      term_off[t] = p;
      first_occ[t] = occ[i];
    }
    if (i == n - 1) {
      term_off[t + 1] = p + 1;
      pstart[p + 1] = (uint32_t)n;
    }
  }
}

__global__ void text_tf_kernel(const uint32_t *pstart, u64 n_postings, uint32_t *tfs) {
  for (u64 p = (u64)blockIdx.x * blockDim.x + threadIdx.x; p < n_postings; p += (u64)gridDim.x * blockDim.x)
    tfs[p] = pstart[p + 1] - pstart[p];
}

// vlen[t] = byte length of term t; vlen[n_terms] = 0 (the scan turns vlen into the vocabulary offsets)
__global__ void text_vocab_len_kernel(const uint32_t *first_occ, const u64 *occ_off, uint32_t n_terms, u64 *vlen) {
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t <= n_terms; t += gridDim.x * blockDim.x)
    vlen[t] = t < n_terms ? occ_off[first_occ[t] + 1] - occ_off[first_occ[t]] : 0;
}

__global__ void text_vocab_copy_kernel(const uint32_t *first_occ, const u64 *occ_off, const uint8_t *arena,
                                       const u64 *vocab_off, uint32_t n_terms, uint8_t *vocab) {
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n_terms; t += gridDim.x * blockDim.x) {
    const uint8_t *src = arena + occ_off[first_occ[t]];
    const u64 n = vocab_off[t + 1] - vocab_off[t];
    for (u64 i = 0; i < n; ++i) vocab[vocab_off[t] + i] = src[i];
  }
}

// ---- vocabulary union (oi_index_bm25_union_vocabulary)
// one thread per entry: the first entry that is empty or holds a byte outside [0-9a-z] -> *bad
__global__ void union_check_kernel(const uint8_t *bytes, const u64 *off, u64 n, unsigned long long *bad) {
  for (u64 e = (u64)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (u64)gridDim.x * blockDim.x) {
    const u64 a = off[e], b = off[e + 1];
    bool ok = b > a;
    for (u64 i = a; ok && i < b; ++i) {
      const uint8_t c = bytes[i];
      ok = (c >= '0' && c <= '9') || (c >= 'a' && c <= 'z');
    }
    if (!ok) atomicMin(bad, (unsigned long long)e);
  }
}

// sorted entry i -> 1 when it starts a term of the union
__global__ void union_flags_kernel(const u64 *keys, const uint32_t *order, const uint8_t *bytes, const u64 *off, u64 n,
                                   uint32_t *flags) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    flags[i] = i == 0 || !same_as_previous(keys, order, bytes, off, i);
}

// scanned flags -> the first entry of every union term
__global__ void union_first_kernel(const uint32_t *scan, const uint32_t *order, u64 n, uint32_t *first) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    if (i == 0 || scan[i] != scan[i - 1]) first[scan[i] - 1] = order[i];
}

// byte order of x[0 .. lx) and y[0 .. ly), a proper prefix first: < 0, 0, > 0
__device__ int bytes_cmp(const uint8_t *x, u64 lx, const uint8_t *y, u64 ly) {
  const u64 n = lx < ly ? lx : ly;
  for (u64 i = 0; i < n; ++i)
    if (x[i] != y[i]) return x[i] < y[i] ? -1 : 1;
  return lx < ly ? -1 : (lx > ly ? 1 : 0);
}

// one thread per local term t: binary search of its bytes in the union -> lens[global id] = its list length; a term the
// union lacks -> *missing
__global__ void union_map_kernel(const uint8_t *lv, const u64 *lv_off, const u64 *term_off, uint32_t n_local,
                                 const uint8_t *uv, const u64 *uv_off, uint32_t n_union, u64 *lens,
                                 unsigned long long *missing) {
  for (uint32_t t = blockIdx.x * blockDim.x + threadIdx.x; t < n_local; t += gridDim.x * blockDim.x) {
    const uint8_t *x = lv + lv_off[t];
    const u64 lx = lv_off[t + 1] - lv_off[t];
    uint32_t lo = 0, hi = n_union;  // first union term >= x
    while (lo < hi) {
      const uint32_t mid = lo + (hi - lo) / 2;
      if (bytes_cmp(uv + uv_off[mid], uv_off[mid + 1] - uv_off[mid], x, lx) < 0) lo = mid + 1; else hi = mid;
    }
    if (lo < n_union && bytes_cmp(uv + uv_off[lo], uv_off[lo + 1] - uv_off[lo], x, lx) == 0)
      lens[lo] = term_off[t + 1] - term_off[t];
    else
      atomicMin(missing, (unsigned long long)t);
  }
}

// cub temporary storage: one buffer, grown when a call needs more
struct CubTmp {
  void *p = nullptr;
  size_t cap = 0;
  CubTmp() = default;
  CubTmp(const CubTmp &) = delete;
  CubTmp &operator=(const CubTmp &) = delete;
  ~CubTmp() { cudaFree(p); }
  cudaError_t reserve(size_t bytes, cudaStream_t st) {
    if (bytes <= cap) return cudaSuccess;
    cudaError_t e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) return e;
    cudaFree(p);
    p = nullptr;
    cap = 0;
    e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
};

// Step 4, shared by the text build (token occurrences) and the vocabulary union (vocabulary entries): sorts the records
// r < n, r = arena[off[r] .. off[r + 1]) with bytes in [0-9a-z] and n < 2^32 - 1, into ascending byte order (a proper
// prefix first), stably.  After run(), keys[i] / order[i] are the key and the record of the i-th place; records with
// the same bytes are neighbours (same_as_previous).  The buffers are freed with the object.
struct RecordSort {
  const u64 *keys = nullptr;
  uint32_t *order = nullptr;
  u64 *d_keys = nullptr, *d_keys2 = nullptr;
  uint32_t *d_vals = nullptr, *d_vals2 = nullptr, *d_pos = nullptr, *d_sub = nullptr, *d_nsel = nullptr;
  RecordSort() = default;
  RecordSort(const RecordSort &) = delete;
  RecordSort &operator=(const RecordSort &) = delete;
  ~RecordSort() {
    cudaFree(d_keys); cudaFree(d_keys2); cudaFree(d_vals); cudaFree(d_vals2); cudaFree(d_pos); cudaFree(d_sub); cudaFree(d_nsel);
  }

  cudaError_t run(const uint8_t *arena, const u64 *off, u64 n, CubTmp &tmp, cudaStream_t st, int num_sms, uint64_t &launches) {
#define RS_CK(call)                     \
  do {                                  \
    const cudaError_t e_ = (call);      \
    if (e_ != cudaSuccess) return e_;   \
  } while (0)
    size_t tb = 0;
    RS_CK(cudaMalloc(&d_keys, n * sizeof(u64)));
    RS_CK(cudaMalloc(&d_keys2, n * sizeof(u64)));
    RS_CK(cudaMalloc(&d_vals, n * sizeof(uint32_t)));
    RS_CK(cudaMalloc(&d_vals2, n * sizeof(uint32_t)));
    text_keys_kernel<<<oi_grid(n, 256, num_sms), 256, 0, st>>>(arena, off, n, d_keys, d_vals);
    ++launches;
    RS_CK(cudaGetLastError());
    cub::DoubleBuffer<u64> kb(d_keys, d_keys2);
    cub::DoubleBuffer<uint32_t> vb(d_vals, d_vals2);
    RS_CK(cub::DeviceRadixSort::SortPairs(nullptr, tb, kb, vb, (int64_t)n, 0, 63, st));
    RS_CK(tmp.reserve(tb, st));
    RS_CK(cub::DeviceRadixSort::SortPairs(tmp.p, tb, kb, vb, (int64_t)n, 0, 63, st));
    launches += 9;  // histogram + one pass per 8 bits
    keys = kb.Current();
    order = vb.Current();
    RS_CK(cudaMalloc(&d_pos, n * sizeof(uint32_t)));
    RS_CK(cudaMalloc(&d_nsel, sizeof(uint32_t)));
    {
      thrust::counting_iterator<uint32_t> idx(0);
      const KeyMayCollide pred{keys};
      RS_CK(cub::DeviceSelect::If(nullptr, tb, idx, d_pos, d_nsel, (int64_t)n, pred, st));
      RS_CK(tmp.reserve(tb, st));
      RS_CK(cub::DeviceSelect::If(tmp.p, tb, idx, d_pos, d_nsel, (int64_t)n, pred, st));
      launches += 2;
    }
    uint32_t m = 0;
    RS_CK(cudaMemcpyAsync(&m, d_nsel, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    RS_CK(cudaStreamSynchronize(st));
    if (m) {
      RS_CK(cudaMalloc(&d_sub, (size_t)m * sizeof(uint32_t)));
      gather_kernel<<<oi_grid(m, 256, num_sms), 256, 0, st>>>(order, d_pos, m, d_sub);
      ++launches;
      RS_CK(cudaGetLastError());
      const TokenLess less{arena, off};
      RS_CK(cub::DeviceMergeSort::StableSortKeys(nullptr, tb, d_sub, (int64_t)m, less, st));
      RS_CK(tmp.reserve(tb, st));
      RS_CK(cub::DeviceMergeSort::StableSortKeys(tmp.p, tb, d_sub, (int64_t)m, less, st));
      launches += 3;  // partition + block sort + merge passes (counted once)
      // the selected slots hold whole runs of equal keys, in key order: the full-byte order refines it in place
      scatter_kernel<<<oi_grid(m, 256, num_sms), 256, 0, st>>>(d_sub, d_pos, m, order);
      ++launches;
      RS_CK(cudaGetLastError());
    }
    return cudaSuccess;
#undef RS_CK
  }
};

}  // namespace

extern "C" oi_status oi_index_build_bm25_text(oi_index *h, const uint8_t *texts, const uint64_t *offsets, uint64_t n_posts,
                                              uint32_t *out_n_terms, uint64_t *out_vocab_bytes) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  {
    const cudaError_t e = cudaSetDevice(h->desc.device);
    if (e != cudaSuccess) return h->fail(OI_ERR_CUDA, "cudaSetDevice failed: %s", cudaGetErrorString(e));
  }
  oi_bm25_free(h);  // from here on, every failure leaves the index without a BM25 part
  if (!texts || !offsets || !out_n_terms || !out_vocab_bytes) return h->fail(OI_ERR_INVALID_ARG, "NULL texts / offsets / output pointer");
  if (n_posts != h->desc.n_docs)
    return h->fail(OI_ERR_INVALID_ARG, "n_posts (%llu) must equal the shard's n_docs (%llu)", (unsigned long long)n_posts,
                   (unsigned long long)h->desc.n_docs);
  for (uint64_t i = 0; i < n_posts; ++i)
    if (offsets[i + 1] < offsets[i]) return h->fail(OI_ERR_INVALID_ARG, "offsets decrease at post %llu", (unsigned long long)i);
  const u64 n_bytes = offsets[n_posts] - offsets[0];
  const u64 n = n_posts;
  cudaStream_t st = h->stream;

  uint8_t *d_text = nullptr, *d_arena = nullptr, *d_vocab = nullptr;
  u64 *d_off = nullptr, *d_tok = nullptr, *d_chr = nullptr, *d_occ_off = nullptr;
  u64 *d_flags = nullptr, *d_term_off = nullptr, *d_vocab_off = nullptr;
  uint32_t *d_doc_len = nullptr, *d_occ_doc = nullptr;
  uint32_t *d_doc_ids = nullptr, *d_tfs = nullptr, *d_pstart = nullptr, *d_first = nullptr;
  CubTmp tmp;
  RecordSort sorted;
  // the CSR arrays and the vocabulary are handed over on success; everything else is freed on every exit
  auto release = [&](bool all) {
    cudaFree(d_text); cudaFree(d_arena); cudaFree(d_off); cudaFree(d_tok); cudaFree(d_chr); cudaFree(d_occ_off);
    cudaFree(d_flags); cudaFree(d_occ_doc); cudaFree(d_pstart); cudaFree(d_first);
    if (all) {
      cudaFree(d_doc_len); cudaFree(d_term_off); cudaFree(d_doc_ids); cudaFree(d_tfs); cudaFree(d_vocab); cudaFree(d_vocab_off);
    }
  };
#define TX_CK(call)                                                                                                   \
  do {                                                                                                                \
    cudaError_t e_ = (call);                                                                                          \
    if (e_ != cudaSuccess) {                                                                                          \
      cudaStreamSynchronize(st);                                                                                      \
      release(true);                                                                                                  \
      return h->fail(e_ == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, "%s failed: %s", #call,   \
                     cudaGetErrorString(e_));                                                                         \
    }                                                                                                                 \
  } while (0)
  size_t tb = 0;

  // ---- 1-2: count pass, scans
  TX_CK(cudaMalloc(&d_text, n_bytes ? n_bytes : 1));
  TX_CK(cudaMalloc(&d_off, (n + 1) * sizeof(u64)));
  TX_CK(cudaMalloc(&d_tok, (n + 1) * sizeof(u64)));
  TX_CK(cudaMalloc(&d_chr, (n + 1) * sizeof(u64)));
  TX_CK(cudaMalloc(&d_doc_len, (n ? n : 1) * sizeof(uint32_t)));
  if (n_bytes) TX_CK(cudaMemcpyAsync(d_text, texts + offsets[0], n_bytes, cudaMemcpyHostToDevice, st));
  TX_CK(cudaMemcpyAsync(d_off, offsets, (n + 1) * sizeof(u64), cudaMemcpyHostToDevice, st));
  TX_CK(cudaMemsetAsync(d_tok + n, 0, sizeof(u64), st));
  TX_CK(cudaMemsetAsync(d_chr + n, 0, sizeof(u64), st));
  u64 warp_blocks = (n + 7) / 8;
  if (warp_blocks > (u64)h->num_sms * 8) warp_blocks = (u64)h->num_sms * 8;
  if (!warp_blocks) warp_blocks = 1;
  // the device offsets are absolute: the kernels see the text through a pointer rebased by offsets[0]
  const uint8_t *d_texts = d_text - offsets[0];
  text_tokens_kernel<false><<<(unsigned)warp_blocks, 256, 0, st>>>(d_texts, d_off, n, d_tok, d_chr, d_doc_len, nullptr, nullptr, nullptr);
  ++h->launches;
  TX_CK(cudaGetLastError());
  TX_CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_tok, d_tok, n + 1, st));
  TX_CK(tmp.reserve(tb, st));
  TX_CK(cub::DeviceScan::ExclusiveSum(tmp.p, tb, d_tok, d_tok, n + 1, st));
  TX_CK(cub::DeviceScan::ExclusiveSum(tmp.p, tb, d_chr, d_chr, n + 1, st));
  h->launches += 4;  // a cub scan = init + scan kernel
  u64 totals[2] = {0, 0};
  TX_CK(cudaMemcpyAsync(&totals[0], d_tok + n, sizeof(u64), cudaMemcpyDeviceToHost, st));
  TX_CK(cudaMemcpyAsync(&totals[1], d_chr + n, sizeof(u64), cudaMemcpyDeviceToHost, st));
  TX_CK(cudaStreamSynchronize(st));
  const u64 T = totals[0], A = totals[1];
  if (T == 0) {
    release(true);
    return h->fail(OI_ERR_INVALID_ARG, "the posts hold no token: an index needs at least one term");
  }
  if (T >= 0xFFFFFFFFull) {
    release(true);
    return h->fail(OI_ERR_INVALID_ARG, "%llu token occurrences: at most 2^32 - 2 per shard", (unsigned long long)T);
  }

  // ---- 3: emit pass
  TX_CK(cudaMalloc(&d_arena, A));
  TX_CK(cudaMalloc(&d_occ_off, (T + 1) * sizeof(u64)));
  TX_CK(cudaMalloc(&d_occ_doc, T * sizeof(uint32_t)));
  TX_CK(cudaMemcpyAsync(d_occ_off + T, &A, sizeof(u64), cudaMemcpyHostToDevice, st));
  text_tokens_kernel<true><<<(unsigned)warp_blocks, 256, 0, st>>>(d_texts, d_off, n, d_tok, d_chr, nullptr, d_arena, d_occ_off, d_occ_doc);
  ++h->launches;
  TX_CK(cudaGetLastError());

  // ---- 4: keys, radix sort, exact order of the tokens that share a key
  TX_CK(sorted.run(d_arena, d_occ_off, T, tmp, st, h->num_sms, h->launches));
  const u64 *keys = sorted.keys;
  const uint32_t *occ = sorted.order;

  // ---- 5: boundaries -> CSR + vocabulary
  TX_CK(cudaMalloc(&d_flags, T * sizeof(u64)));
  text_flags_kernel<<<oi_grid(T, 256, h->num_sms), 256, 0, st>>>(keys, occ, d_arena, d_occ_off, d_occ_doc, T, d_flags);
  ++h->launches;
  TX_CK(cudaGetLastError());
  TX_CK(cub::DeviceScan::InclusiveSum(nullptr, tb, d_flags, d_flags, (int64_t)T, st));
  TX_CK(tmp.reserve(tb, st));
  TX_CK(cub::DeviceScan::InclusiveSum(tmp.p, tb, d_flags, d_flags, (int64_t)T, st));
  h->launches += 2;
  u64 last = 0;
  TX_CK(cudaMemcpyAsync(&last, d_flags + T - 1, sizeof(u64), cudaMemcpyDeviceToHost, st));
  TX_CK(cudaStreamSynchronize(st));
  const uint32_t V = (uint32_t)(last >> 32);
  const u64 P = (uint32_t)last;
  TX_CK(cudaMalloc(&d_term_off, ((size_t)V + 1) * sizeof(u64)));
  TX_CK(cudaMalloc(&d_doc_ids, P * sizeof(uint32_t)));
  TX_CK(cudaMalloc(&d_tfs, P * sizeof(uint32_t)));
  TX_CK(cudaMalloc(&d_pstart, (P + 1) * sizeof(uint32_t)));
  TX_CK(cudaMalloc(&d_first, (size_t)V * sizeof(uint32_t)));
  text_csr_kernel<<<oi_grid(T, 256, h->num_sms), 256, 0, st>>>(d_flags, occ, d_occ_doc, T, d_term_off, d_doc_ids, d_pstart, d_first);
  text_tf_kernel<<<oi_grid(P, 256, h->num_sms), 256, 0, st>>>(d_pstart, P, d_tfs);
  h->launches += 2;
  TX_CK(cudaGetLastError());
  TX_CK(cudaMalloc(&d_vocab_off, ((size_t)V + 1) * sizeof(u64)));
  text_vocab_len_kernel<<<oi_grid((u64)V + 1, 256, h->num_sms), 256, 0, st>>>(d_first, d_occ_off, V, d_vocab_off);
  ++h->launches;
  TX_CK(cudaGetLastError());
  TX_CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_vocab_off, d_vocab_off, (int64_t)V + 1, st));
  TX_CK(tmp.reserve(tb, st));
  TX_CK(cub::DeviceScan::ExclusiveSum(tmp.p, tb, d_vocab_off, d_vocab_off, (int64_t)V + 1, st));
  h->launches += 2;
  u64 vocab_bytes = 0;
  TX_CK(cudaMemcpyAsync(&vocab_bytes, d_vocab_off + V, sizeof(u64), cudaMemcpyDeviceToHost, st));
  TX_CK(cudaStreamSynchronize(st));
  TX_CK(cudaMalloc(&d_vocab, vocab_bytes));
  text_vocab_copy_kernel<<<oi_grid(V, 256, h->num_sms), 256, 0, st>>>(d_first, d_occ_off, d_arena, d_vocab_off, V, d_vocab);
  ++h->launches;
  TX_CK(cudaGetLastError());
  TX_CK(cudaStreamSynchronize(st));
#undef TX_CK

  // ---- 6: hand-off
  release(false);
  const oi_status s = oi_bm25_adopt(h, V, P, d_term_off, d_doc_ids, d_tfs, d_doc_len);
  if (s != OI_OK) {
    cudaFree(d_vocab);
    cudaFree(d_vocab_off);
    return s;
  }
  h->d_vocab = d_vocab;
  h->d_vocab_off = d_vocab_off;
  h->vocab_bytes = vocab_bytes;
  *out_n_terms = V;
  *out_vocab_bytes = vocab_bytes;
  return OI_OK;
}

// The document-sharded lift: the shards' vocabularies, gathered by the host, become one sorted union (the entries go
// through step 4 as records, then the boundary flags of step 5 and the vocabulary assembly), and this shard's lists are
// re-indexed to it (one binary search per local term, an exclusive scan of the list lengths).  The postings do not
// move: the map from local to global term ids is strictly increasing.  Every new array is built next to the old ones
// and swapped in at the end, so a failed call leaves the BM25 part as it was.
extern "C" oi_status oi_index_bm25_union_vocabulary(oi_index *h, const uint8_t *terms, const uint64_t *offsets,
                                                    uint64_t n_entries, uint32_t *out_n_terms, uint64_t *out_vocab_bytes) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  if (!terms || !offsets || !out_n_terms || !out_vocab_bytes) return h->fail(OI_ERR_INVALID_ARG, "NULL terms / offsets / output pointer");
  if (n_entries == 0) return h->fail(OI_ERR_INVALID_ARG, "no entries: the union needs at least this shard's terms");
  if (n_entries >= 0xFFFFFFFFull)
    return h->fail(OI_ERR_INVALID_ARG, "%llu entries: at most 2^32 - 2", (unsigned long long)n_entries);
  const u64 *term_off = oi_bm25_term_offsets(h);
  if (!term_off || !h->d_vocab_off) return h->fail(OI_ERR_STATE, "the BM25 part was not built from text: no vocabulary to unite");
  if (oi_bm25_finalized(h)) return h->fail(OI_ERR_STATE, "the BM25 part is finalized: unite the vocabularies before oi_index_bm25_finalize");
  for (uint64_t i = 0; i < n_entries; ++i)
    if (offsets[i + 1] < offsets[i]) return h->fail(OI_ERR_INVALID_ARG, "offsets decrease at entry %llu", (unsigned long long)i);
  {
    const cudaError_t e = cudaSetDevice(h->desc.device);
    if (e != cudaSuccess) return h->fail(OI_ERR_CUDA, "cudaSetDevice failed: %s", cudaGetErrorString(e));
  }
  const u64 n = n_entries, n_bytes = offsets[n_entries] - offsets[0];
  const uint32_t n_local = oi_bm25_n_terms(h);
  cudaStream_t st = h->stream;

  uint8_t *d_bytes = nullptr, *d_vocab = nullptr;
  u64 *d_off = nullptr, *d_vocab_off = nullptr, *d_term_off = nullptr;
  uint32_t *d_flags = nullptr, *d_first = nullptr;
  unsigned long long *d_err = nullptr;
  CubTmp tmp;
  RecordSort sorted;
  // the new vocabulary and term offsets are handed over on success; everything else is freed on every exit
  auto release = [&](bool all) {
    cudaFree(d_bytes); cudaFree(d_off); cudaFree(d_flags); cudaFree(d_first); cudaFree(d_err);
    if (all) {
      cudaFree(d_vocab); cudaFree(d_vocab_off); cudaFree(d_term_off);
    }
  };
#define UN_CK(call)                                                                                                   \
  do {                                                                                                                \
    cudaError_t e_ = (call);                                                                                          \
    if (e_ != cudaSuccess) {                                                                                          \
      cudaStreamSynchronize(st);                                                                                      \
      release(true);                                                                                                  \
      return h->fail(e_ == cudaErrorMemoryAllocation ? OI_ERR_OUT_OF_MEMORY : OI_ERR_CUDA, "%s failed: %s", #call,   \
                     cudaGetErrorString(e_));                                                                         \
    }                                                                                                                 \
  } while (0)
  size_t tb = 0;

  // ---- the entries: copy, check (empty entries and bytes outside [0-9a-z] come from other processes)
  UN_CK(cudaMalloc(&d_bytes, n_bytes ? n_bytes : 1));
  UN_CK(cudaMalloc(&d_off, (n + 1) * sizeof(u64)));
  UN_CK(cudaMalloc(&d_err, 2 * sizeof(unsigned long long)));
  if (n_bytes) UN_CK(cudaMemcpyAsync(d_bytes, terms + offsets[0], n_bytes, cudaMemcpyHostToDevice, st));
  UN_CK(cudaMemcpyAsync(d_off, offsets, (n + 1) * sizeof(u64), cudaMemcpyHostToDevice, st));
  UN_CK(cudaMemsetAsync(d_err, 0xFF, 2 * sizeof(unsigned long long), st));
  // the device offsets are absolute: the kernels see the entries through a pointer rebased by offsets[0]
  const uint8_t *d_terms = d_bytes - offsets[0];
  union_check_kernel<<<oi_grid(n, 256, h->num_sms), 256, 0, st>>>(d_terms, d_off, n, d_err);
  ++h->launches;
  UN_CK(cudaGetLastError());
  unsigned long long bad = 0;
  UN_CK(cudaMemcpyAsync(&bad, d_err, sizeof(bad), cudaMemcpyDeviceToHost, st));
  UN_CK(cudaStreamSynchronize(st));
  if (bad != ~0ull) {
    release(true);
    return h->fail(OI_ERR_INVALID_ARG, "entry %llu is empty or holds a byte outside [0-9a-z]", bad);
  }

  // ---- union: byte order (step 4), boundaries, vocabulary
  UN_CK(sorted.run(d_terms, d_off, n, tmp, st, h->num_sms, h->launches));
  UN_CK(cudaMalloc(&d_flags, n * sizeof(uint32_t)));
  union_flags_kernel<<<oi_grid(n, 256, h->num_sms), 256, 0, st>>>(sorted.keys, sorted.order, d_terms, d_off, n, d_flags);
  ++h->launches;
  UN_CK(cudaGetLastError());
  UN_CK(cub::DeviceScan::InclusiveSum(nullptr, tb, d_flags, d_flags, (int64_t)n, st));
  UN_CK(tmp.reserve(tb, st));
  UN_CK(cub::DeviceScan::InclusiveSum(tmp.p, tb, d_flags, d_flags, (int64_t)n, st));
  h->launches += 2;
  uint32_t V = 0;
  UN_CK(cudaMemcpyAsync(&V, d_flags + n - 1, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  UN_CK(cudaStreamSynchronize(st));
  UN_CK(cudaMalloc(&d_first, (size_t)V * sizeof(uint32_t)));
  union_first_kernel<<<oi_grid(n, 256, h->num_sms), 256, 0, st>>>(d_flags, sorted.order, n, d_first);
  ++h->launches;
  UN_CK(cudaGetLastError());
  UN_CK(cudaMalloc(&d_vocab_off, ((size_t)V + 1) * sizeof(u64)));
  text_vocab_len_kernel<<<oi_grid((u64)V + 1, 256, h->num_sms), 256, 0, st>>>(d_first, d_off, V, d_vocab_off);
  ++h->launches;
  UN_CK(cudaGetLastError());
  UN_CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_vocab_off, d_vocab_off, (int64_t)V + 1, st));
  UN_CK(tmp.reserve(tb, st));
  UN_CK(cub::DeviceScan::ExclusiveSum(tmp.p, tb, d_vocab_off, d_vocab_off, (int64_t)V + 1, st));
  h->launches += 2;
  u64 vocab_bytes = 0;
  UN_CK(cudaMemcpyAsync(&vocab_bytes, d_vocab_off + V, sizeof(u64), cudaMemcpyDeviceToHost, st));
  UN_CK(cudaStreamSynchronize(st));
  UN_CK(cudaMalloc(&d_vocab, vocab_bytes));
  text_vocab_copy_kernel<<<oi_grid(V, 256, h->num_sms), 256, 0, st>>>(d_first, d_off, d_terms, d_vocab_off, V, d_vocab);
  ++h->launches;
  UN_CK(cudaGetLastError());

  // ---- this shard's lists under the global term ids: lengths scattered to their global ids, exclusive scan
  UN_CK(cudaMalloc(&d_term_off, ((size_t)V + 1) * sizeof(u64)));
  UN_CK(cudaMemsetAsync(d_term_off, 0, ((size_t)V + 1) * sizeof(u64), st));
  union_map_kernel<<<oi_grid(n_local, 256, h->num_sms), 256, 0, st>>>(h->d_vocab, h->d_vocab_off, term_off, n_local, d_vocab,
                                                                  d_vocab_off, V, d_term_off, d_err + 1);
  ++h->launches;
  UN_CK(cudaGetLastError());
  UN_CK(cub::DeviceScan::ExclusiveSum(nullptr, tb, d_term_off, d_term_off, (int64_t)V + 1, st));
  UN_CK(tmp.reserve(tb, st));
  UN_CK(cub::DeviceScan::ExclusiveSum(tmp.p, tb, d_term_off, d_term_off, (int64_t)V + 1, st));
  h->launches += 2;
  unsigned long long missing = 0;
  UN_CK(cudaMemcpyAsync(&missing, d_err + 1, sizeof(missing), cudaMemcpyDeviceToHost, st));
  UN_CK(cudaStreamSynchronize(st));
  if (missing != ~0ull) {
    // name the term: its bytes are read back from this shard's vocabulary
    u64 span[2] = {0, 0};
    char term[65] = {0};
    UN_CK(cudaMemcpyAsync(span, h->d_vocab_off + missing, sizeof(span), cudaMemcpyDeviceToHost, st));
    UN_CK(cudaStreamSynchronize(st));
    const u64 len = span[1] - span[0] < 64 ? span[1] - span[0] : 64;
    UN_CK(cudaMemcpyAsync(term, h->d_vocab + span[0], len, cudaMemcpyDeviceToHost, st));
    UN_CK(cudaStreamSynchronize(st));
    release(true);
    return h->fail(OI_ERR_INVALID_ARG, "term %llu of this shard (\"%s%s\") is missing from the entries", missing, term,
                   span[1] - span[0] > 64 ? "..." : "");
  }
#undef UN_CK

  // ---- hand-off: nothing below can fail
  release(false);
  cudaFree(h->d_vocab);
  cudaFree(h->d_vocab_off);
  h->d_vocab = d_vocab;
  h->d_vocab_off = d_vocab_off;
  h->vocab_bytes = vocab_bytes;
  oi_bm25_replace_terms(h, V, d_term_off);
  *out_n_terms = V;
  *out_vocab_bytes = vocab_bytes;
  return OI_OK;
}

extern "C" oi_status oi_index_read_vocabulary(oi_index *h, uint8_t *bytes, uint64_t *offsets) {
  if (!h) return OI_ERR_INVALID_ARG;
  std::lock_guard<std::mutex> lock(h->mu);
  if (!h->d_vocab_off) return h->fail(OI_ERR_STATE, "the BM25 part was not built from text: no vocabulary");
  if (!bytes || !offsets) return h->fail(OI_ERR_INVALID_ARG, "NULL bytes / offsets");
  cudaError_t e = cudaSetDevice(h->desc.device);
  if (e == cudaSuccess) e = cudaMemcpyAsync(bytes, h->d_vocab, h->vocab_bytes, cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess)
    e = cudaMemcpyAsync(offsets, h->d_vocab_off, ((size_t)oi_bm25_n_terms(h) + 1) * sizeof(u64), cudaMemcpyDeviceToHost, h->stream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->stream);
  if (e != cudaSuccess) return h->fail(OI_ERR_CUDA, "reading the vocabulary failed: %s", cudaGetErrorString(e));
  return OI_OK;
}
