"""ctypes binding of include/openintel_gpu.h.  Mirrors the C ABI one to one; every non-zero
status raises OiError carrying oi_last_error().  The library must exist: a missing .so is a
hard error (the product has no CPU path)."""
import ctypes as C
import os

import numpy as np

NO_DOC = 0xFFFFFFFF
DTYPE_F32, DTYPE_BF16 = 0, 1
UNIQUE_ID_BYTES = 128
P2P_HANDLE_BYTES = 64
_HERE = os.path.dirname(os.path.abspath(__file__))

STATUS_NAMES = {1: "INVALID_ARG", 2: "NO_DEVICE", 3: "CUDA", 4: "OUT_OF_MEMORY", 5: "STATE", 6: "COMM", 7: "UNSUPPORTED"}


class OiError(RuntimeError):
    def __init__(self, status, message):
        super().__init__("openintel_gpu: %s (%d): %s" % (STATUS_NAMES.get(status, "?"), status, message))
        self.status = status
        self.message = message


class IndexDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("device", C.c_int32), ("n_docs", C.c_uint64),
                ("doc_base", C.c_uint64), ("dim", C.c_uint32), ("dtype", C.c_uint32),
                ("max_k", C.c_uint32), ("max_batch", C.c_uint32)]


class Bm25Params(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("k1", C.c_float), ("b", C.c_float), ("avgdl", C.c_float),
                ("n_docs_global", C.c_uint64), ("global_df", C.POINTER(C.c_uint32))]


class SocialSummary(C.Structure):
    """oi_social_summary: SpeculationEngine::social_summary of a batch (src/domain/engine/speculation_engine.rs:70-125)"""
    _fields_ = [("total", C.c_uint64), ("bullish", C.c_uint64), ("bearish", C.c_uint64), ("neutral", C.c_uint64),
                ("net_sentiment", C.c_double), ("speculation_index", C.c_double), ("bull_bear_ratio", C.c_double)]


N_SOURCES = 2  # OI_N_SOURCES: post sources in store-schema order (store.SOURCES)


def _source_code(source):
    """a mention call's source argument: -1 for all posts (None), else the source code"""
    return -1 if source is None else int(source)


# oi_mention_state as a numpy structured type: the running state of one term's summary after a prefix of the doc order
# (SPEC §8a)
MENTION_STATE_DTYPE = np.dtype([("total", "<u8"), ("bullish", "<u8"), ("bearish", "<u8"), ("neutral", "<u8"),
                                ("speculative", "<u8"), ("by_source", "<u8", (N_SOURCES,)), ("sum", "<f8")])
# ... and of oi_social_summary
SOCIAL_SUMMARY_DTYPE = np.dtype([(f, "<u8" if t is C.c_uint64 else "<f8") for f, t in SocialSummary._fields_])


def lib_path():
    # OI_GPU_LIB: A/B experiments against another build of the same C ABI (tools/ only); the product loads the in-tree .so
    return os.environ.get("OI_GPU_LIB") or os.path.join(_HERE, "libopenintel_gpu.so")


_lib = None
_vp, _u32p, _u64p, _f32p = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p  # raw addresses


def load_library():
    """dlopen libopenintel_gpu.so and declare every prototype of include/openintel_gpu.h."""
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise OSError("libopenintel_gpu.so is missing (%s): build it with "
                      "`python -m openintel_b200._build`; there is no CPU fallback" % p)
    L = C.CDLL(p, mode=C.RTLD_GLOBAL)
    st, H = C.c_int32, C.c_void_p
    sig = {
        "oi_index_create": (st, [C.POINTER(IndexDesc), C.POINTER(H)]),
        "oi_index_destroy": (None, [H]),
        "oi_last_error": (C.c_char_p, [H]),
        "oi_version": (C.c_char_p, []),
        "oi_index_load_embeddings": (st, [H, _vp, C.c_uint64, C.c_uint64]),
        "oi_index_synth_embeddings": (st, [H, C.c_uint64]),
        "oi_index_read_embeddings": (st, [H, _vp, C.c_uint64, C.c_uint64]),
        "oi_index_load_bm25": (st, [H, _u64p, _u32p, _u32p, _u32p, C.c_uint32]),
        "oi_index_synth_bm25": (st, [H, C.c_uint64, C.c_uint32, _vp]),
        "oi_index_build_bm25_text": (st, [H, _vp, _u64p, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
        "oi_index_bm25_union_vocabulary": (st, [H, _vp, _u64p, C.c_uint64, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64)]),
        "oi_index_read_vocabulary": (st, [H, _vp, _u64p]),
        "oi_index_bm25_local_stats": (st, [H, _u32p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
        "oi_index_bm25_finalize": (st, [H, C.POINTER(Bm25Params)]),
        "oi_index_read_bm25": (st, [H, _u64p, _u32p, _u32p, _u32p, _f32p]),
        "oi_comm_unique_id": (st, [_vp]),
        "oi_index_comm_init": (st, [H, C.c_int32, C.c_int32, _vp]),
        "oi_index_p2p_export": (st, [H, _vp]),
        "oi_index_p2p_attach": (st, [H, _vp]),
        "oi_index_p2p_status": (st, [H, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
        "oi_search_cosine": (st, [H, _f32p, C.c_uint32, C.c_uint32, _u32p, _f32p]),
        "oi_search_bm25": (st, [H, _u32p, _u32p, C.c_uint32, C.c_uint32, _u32p, _f32p]),
        "oi_search_hybrid": (st, [H, _f32p, _u32p, _u32p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, _f32p, _u32p, _u32p]),
        "oi_search_cosine_dev": (st, [H, _f32p, C.c_uint32, C.c_uint32, _u32p, _f32p, _vp]),
        "oi_search_bm25_dev": (st, [H, _u32p, _u32p, C.c_uint32, C.c_uint32, _u32p, _f32p, _vp]),
        "oi_search_hybrid_dev": (st, [H, _f32p, _u32p, _u32p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, _f32p, _u32p, _u32p, _vp]),
        "oi_lexicon_analyze": (st, [C.c_int32, _vp, _u64p, C.c_uint64, _vp, _vp, _u32p, _u32p]),
        "oi_lexicon_create": (st, [C.c_int32, C.c_uint64, C.c_uint64, C.POINTER(H)]),
        "oi_lexicon_destroy": (None, [H]),
        "oi_lexicon_run": (st, [H, _vp, _u64p, C.c_uint64, _vp, _vp, _u32p, _u32p, C.c_double, C.POINTER(SocialSummary)]),
        "oi_lexicon_launch_count": (C.c_uint64, [H]),
        "oi_index_load_post_signals": (st, [H, _vp, _vp, _vp]),
        "oi_index_mention_summary": (st, [H, _u32p, C.c_uint32, C.c_int32, C.c_double, _vp, _vp, _vp]),
        "oi_index_load_post_times": (st, [H, _vp]),
        "oi_index_mention_timeline": (st, [H, _u32p, C.c_uint32, _vp, C.c_uint32, C.c_int32, C.c_double, _vp, _vp, _vp]),
        "oi_index_mention_counts": (st, [H, _vp, C.c_uint32, C.c_int32, _u32p]),
        "oi_index_launch_count": (C.c_uint64, [H]),
        "oi_index_set_option": (st, [H, C.c_char_p, C.c_int64]),
        "oi_debug_cosine_gemm_scores": (st, [H, _f32p, C.c_uint32, _f32p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError here = the .so does not export what the header declares
        fn.restype, fn.argtypes = res, args
    L._oi_sig = sig
    _lib = L
    return L


def version():
    return load_library().oi_version().decode()


def _addr(a):
    """address of a numpy array / torch tensor / int / None"""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"]
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


class GpuIndex:
    """One shard on one GPU (wraps an oi_index*)."""

    def __init__(self, n_docs, dim, dtype=DTYPE_F32, device=0, doc_base=0, max_k=100, max_batch=1):
        self.L = load_library()
        self.n_docs, self.dim, self.dtype, self.doc_base = int(n_docs), int(dim), int(dtype), int(doc_base)
        self.max_k, self.max_batch = int(max_k), int(max_batch)
        d = IndexDesc(C.sizeof(IndexDesc), device, n_docs, doc_base, dim, dtype, max_k, max_batch)
        self.h = C.c_void_p()
        s = self.L.oi_index_create(C.byref(d), C.byref(self.h))
        if s:
            self.h = None
            raise OiError(s, self.L.oi_last_error(None).decode())

    def _ck(self, s):
        if s:
            raise OiError(s, self.L.oi_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.oi_index_destroy(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # -- embeddings
    def np_dtype(self):
        return np.float32 if self.dtype == DTYPE_F32 else np.uint16

    def load_embeddings(self, rows, first_doc=0):
        rows = np.ascontiguousarray(rows, dtype=self.np_dtype())
        assert rows.ndim == 2 and rows.shape[1] == self.dim
        self._ck(self.L.oi_index_load_embeddings(self.h, _addr(rows), first_doc, rows.shape[0]))

    def synth_embeddings(self, seed):
        self._ck(self.L.oi_index_synth_embeddings(self.h, seed))

    def read_embeddings(self, first_doc, n):
        out = np.empty((n, self.dim), dtype=self.np_dtype())
        self._ck(self.L.oi_index_read_embeddings(self.h, _addr(out), first_doc, n))
        return out

    # -- BM25
    def load_bm25(self, term_offsets, doc_ids, tfs, doc_len):
        to = np.ascontiguousarray(term_offsets, dtype=np.uint64)
        di = np.ascontiguousarray(doc_ids, dtype=np.uint32)
        tf = np.ascontiguousarray(tfs, dtype=np.uint32)
        dl = np.ascontiguousarray(doc_len, dtype=np.uint32)
        assert len(dl) == self.n_docs and len(di) == len(tf) == int(to[-1])
        self.n_terms = len(to) - 1
        self._ck(self.L.oi_index_load_bm25(self.h, _addr(to), _addr(di), _addr(tf), _addr(dl), self.n_terms))

    def synth_bm25(self, seed, vocab, zipf_cdf):
        cdf = np.ascontiguousarray(zipf_cdf, dtype=np.float64)
        assert len(cdf) == vocab
        self.n_terms = vocab
        self._ck(self.L.oi_index_synth_bm25(self.h, seed, vocab, _addr(cdf)))

    def build_bm25_text(self, texts):
        """posts (str or bytes, one per document) -> this shard's BM25 part, tokenized and indexed on the device
        (oi_index_build_bm25_text); follow with bm25_finalize.  Returns the vocabulary: term id i = list[i]."""
        blob, offs = pack_texts(texts)
        nt, nb = C.c_uint32(), C.c_uint64()
        self._ck(self.L.oi_index_build_bm25_text(self.h, _addr(blob), _addr(offs), len(offs) - 1, C.byref(nt), C.byref(nb)))
        self.n_terms, self.vocab_bytes = nt.value, nb.value
        return unpack_terms(*self.read_vocabulary_packed())

    def bm25_union_vocabulary(self, blob, offsets):
        """document-sharded index, after build_bm25_text and before bm25_finalize: (blob u8[], offsets u64[n + 1]) = the
        concatenated vocabularies of all shards (any order, duplicates allowed; sharding.all_gather_packed).  The
        vocabulary becomes their sorted union and this shard's lists are re-indexed to it, on the device
        (oi_index_bm25_union_vocabulary).  Returns the global vocabulary: term id i = list[i]."""
        blob = np.ascontiguousarray(blob, dtype=np.uint8)
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        if not len(blob):
            blob = np.zeros(1, dtype=np.uint8)
        nt, nb = C.c_uint32(), C.c_uint64()
        self._ck(self.L.oi_index_bm25_union_vocabulary(self.h, _addr(blob), _addr(offs), len(offs) - 1, C.byref(nt), C.byref(nb)))
        self.n_terms, self.vocab_bytes = nt.value, nb.value
        return unpack_terms(*self.read_vocabulary_packed())

    def read_vocabulary_packed(self):
        """the vocabulary of a BM25 part built from text, undecoded: (bytes u8[], offsets u64[n_terms + 1]), term t =
        bytes[offsets[t] .. offsets[t + 1])"""
        vb = np.empty(max(getattr(self, "vocab_bytes", 0), 1), dtype=np.uint8)
        vo = np.empty(self.n_terms + 1, dtype=np.uint64)
        self._ck(self.L.oi_index_read_vocabulary(self.h, _addr(vb), _addr(vo)))
        return vb[:int(vo[-1])], vo

    def bm25_local_stats(self):
        df = np.empty(self.n_terms, dtype=np.uint32)
        sdl, npost = C.c_uint64(), C.c_uint64()
        self._ck(self.L.oi_index_bm25_local_stats(self.h, _addr(df), C.byref(sdl), C.byref(npost)))
        return df, sdl.value, npost.value

    def bm25_finalize(self, k1=1.2, b=0.75, avgdl=0.0, n_docs_global=0, global_df=None):
        gdf = None if global_df is None else np.ascontiguousarray(global_df, dtype=np.uint32)
        p = Bm25Params(C.sizeof(Bm25Params), k1, b, avgdl, n_docs_global,
                       None if gdf is None else gdf.ctypes.data_as(C.POINTER(C.c_uint32)))
        self._ck(self.L.oi_index_bm25_finalize(self.h, C.byref(p)))

    def read_bm25(self, n_postings):
        to = np.empty(self.n_terms + 1, dtype=np.uint64)
        di = np.empty(n_postings, dtype=np.uint32)
        tf = np.empty(n_postings, dtype=np.uint32)
        dl = np.empty(self.n_docs, dtype=np.uint32)
        w = np.empty(n_postings, dtype=np.float32)
        self._ck(self.L.oi_index_read_bm25(self.h, _addr(to), _addr(di), _addr(tf), _addr(dl), _addr(w)))
        return dict(term_offsets=to, doc_ids=di, tfs=tf, doc_len=dl, weights=w)

    # -- per-term social summaries over the posting lists (SPEC §8a)
    def load_post_signals(self, polarity, speculative, source):
        """per-post lexicon signals of this shard, in doc order: polarity f64 in [-1, 1], speculative 0/1, source code
        (index into store.SOURCES).  A refused call keeps the previous signals."""
        pol = np.ascontiguousarray(polarity, dtype=np.float64)
        spec = np.ascontiguousarray(speculative, dtype=np.uint8)
        src = np.ascontiguousarray(source, dtype=np.uint8)
        if not len(pol) == len(spec) == len(src) == self.n_docs:
            raise ValueError("need %d signals of each kind, got %d / %d / %d" % (self.n_docs, len(pol), len(spec), len(src)))
        self._ck(self.L.oi_index_load_post_signals(self.h, _addr(pol), _addr(spec), _addr(src)))

    def mention_summary(self, term_ids, source=None, threshold=0.2, carry=None):
        """the social summary of each term's posting list on this shard (oi_index_mention_summary), continued from
        `carry` (the states of the previous shard, or None).  source: None = all posts, else a source code.
        -> (states: MENTION_STATE_DTYPE array, summaries: list of dicts shaped like GpuLexicon's summary)"""
        terms = np.ascontiguousarray(term_ids, dtype=np.uint32).reshape(-1)
        states, sums, cin = self._mention_outputs((len(terms),), carry)
        self._ck(self.L.oi_index_mention_summary(self.h, _addr(terms), len(terms), _source_code(source), threshold,
                                                  _addr(cin), _addr(states), _addr(sums)))
        return states, summaries_from_array(sums)

    @staticmethod
    def _mention_outputs(shape, carry):
        """zeroed states and summaries of a mention call, shaped (terms,) or (terms, buckets), and the carried states
        checked against that shape (None when not given)"""
        states = np.zeros(shape, dtype=MENTION_STATE_DTYPE)
        sums = np.zeros(shape, dtype=SOCIAL_SUMMARY_DTYPE)
        cin = None
        if carry is not None:
            cin = np.ascontiguousarray(carry, dtype=MENTION_STATE_DTYPE)
            if cin.size != states.size:
                what = ("%d terms x %d buckets" if len(shape) == 2 else "%d terms") % shape
                raise ValueError("%d carried states for %s" % (cin.size, what))
        return states, sums, cin

    # -- per-term timelines (SPEC §8b)
    def load_post_times(self, seconds):
        """per-post creation times of this shard, in doc order: int64 seconds since the Unix epoch"""
        t = np.ascontiguousarray(seconds, dtype=np.int64)
        if t.ndim != 1 or len(t) != self.n_docs:
            raise ValueError("need %d post times, got %d" % (self.n_docs, t.size))
        self._ck(self.L.oi_index_load_post_times(self.h, _addr(t)))

    def mention_timeline(self, term_ids, edges, source=None, threshold=0.2, carry=None):
        """the social summary of each term's posts in each bucket [edges[b], edges[b + 1]) on this shard
        (oi_index_mention_timeline), continued from `carry` ([n][B] states of the previous shard, or None).
        -> (states: MENTION_STATE_DTYPE [n][B], summaries: n lists of B dicts shaped like GpuLexicon's summary)"""
        terms = np.ascontiguousarray(term_ids, dtype=np.uint32).reshape(-1)
        e = np.ascontiguousarray(edges, dtype=np.int64).reshape(-1)
        n, nb = len(terms), max(len(e) - 1, 0)
        states, sums, cin = self._mention_outputs((n, nb), carry)
        self._ck(self.L.oi_index_mention_timeline(self.h, _addr(terms), n, _addr(e), nb, _source_code(source), threshold,
                                                   _addr(cin), _addr(states), _addr(sums)))
        return states, [summaries_from_array(row) for row in sums]

    # -- per-term mention counts over the whole vocabulary (SPEC §8c)
    def mention_counts(self, edges, source=None):
        """the number of this shard's posts that mention each term of the BM25 part and were created in each bucket
        [edges[b], edges[b + 1]) (oi_index_mention_counts).  -> uint32 [n_terms][B]"""
        e = np.ascontiguousarray(edges, dtype=np.int64).reshape(-1)
        nb = max(len(e) - 1, 0)
        out = np.zeros((getattr(self, "n_terms", 0), nb), dtype=np.uint32)  # no BM25 part: the call refuses
        self._ck(self.L.oi_index_mention_counts(self.h, _addr(e), nb, _source_code(source), _addr(out)))
        return out

    # -- multi-GPU
    @staticmethod
    def comm_unique_id():
        L = load_library()
        buf = np.zeros(UNIQUE_ID_BYTES, dtype=np.uint8)
        s = L.oi_comm_unique_id(_addr(buf))
        if s:
            raise OiError(s, "oi_comm_unique_id failed (NCCL not loadable?)")
        return buf

    def comm_init(self, rank, world, unique_id):
        uid = np.ascontiguousarray(unique_id, dtype=np.uint8)
        self._ck(self.L.oi_index_comm_init(self.h, rank, world, _addr(uid)))

    def p2p_export(self):
        """handle (64 bytes) of this rank's exchange buffer: distribute to every rank, then p2p_attach"""
        buf = np.zeros(P2P_HANDLE_BYTES, dtype=np.uint8)
        self._ck(self.L.oi_index_p2p_export(self.h, _addr(buf)))
        return buf

    def p2p_attach(self, handles):
        hs = np.ascontiguousarray(handles, dtype=np.uint8).reshape(-1, P2P_HANDLE_BYTES)
        self._ck(self.L.oi_index_p2p_attach(self.h, _addr(hs)))

    def p2p_status(self):
        n, bad = C.c_uint64(), C.c_uint32()
        self._ck(self.L.oi_index_p2p_status(self.h, C.byref(n), C.byref(bad)))
        return n.value, bool(bad.value)

    # -- search, host buffers (numpy or pinned torch tensors)
    @staticmethod
    def _pack_terms(q_terms):
        if isinstance(q_terms, tuple):
            return q_terms
        if isinstance(q_terms, np.ndarray) and q_terms.ndim == 2:
            nq, t = q_terms.shape
            return (np.ascontiguousarray(q_terms, dtype=np.uint32).reshape(-1),
                    (np.arange(nq + 1, dtype=np.uint32) * t))
        offs = np.zeros(len(q_terms) + 1, dtype=np.uint32)
        offs[1:] = np.cumsum([len(q) for q in q_terms])
        flat = np.concatenate([np.asarray(q, dtype=np.uint32) for q in q_terms]) if len(q_terms) else np.zeros(0, np.uint32)
        return np.ascontiguousarray(flat, dtype=np.uint32), offs

    def search_cosine(self, queries, k, out_ids=None, out_scores=None):
        if isinstance(queries, np.ndarray):
            queries = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        nq = queries.shape[0]
        if out_ids is None:
            out_ids = np.empty((nq, k), dtype=np.uint32)
            out_scores = np.empty((nq, k), dtype=np.float32)
        self._ck(self.L.oi_search_cosine(self.h, _addr(queries), nq, k, _addr(out_ids), _addr(out_scores)))
        return out_ids, out_scores

    def search_bm25(self, q_terms, k):
        flat, offs = self._pack_terms(q_terms)
        nq = len(offs) - 1
        ids = np.empty((nq, k), dtype=np.uint32)
        sc = np.empty((nq, k), dtype=np.float32)
        self._ck(self.L.oi_search_bm25(self.h, _addr(flat), _addr(offs), nq, k, _addr(ids), _addr(sc)))
        return ids, sc

    def search_hybrid(self, queries, q_terms, k, rrf_k=60):
        queries = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        flat, offs = self._pack_terms(q_terms)
        nq = queries.shape[0]
        assert len(offs) - 1 == nq
        ids = np.empty((nq, k), dtype=np.uint32)
        rrf = np.empty((nq, k), dtype=np.float32)
        rc = np.empty((nq, k), dtype=np.uint32)
        rb = np.empty((nq, k), dtype=np.uint32)
        self._ck(self.L.oi_search_hybrid(self.h, _addr(queries), _addr(flat), _addr(offs), nq, k, rrf_k,
                                         _addr(ids), _addr(rrf), _addr(rc), _addr(rb)))
        return ids, rrf, rc, rb

    # -- search, device-resident (torch CUDA tensors or raw device addresses)
    def search_cosine_dev(self, d_queries, nq, k, d_out_ids, d_out_scores, stream=0):
        self._ck(self.L.oi_search_cosine_dev(self.h, _addr(d_queries), nq, k, _addr(d_out_ids), _addr(d_out_scores), stream))

    def search_bm25_dev(self, d_terms, d_offs, nq, k, d_out_ids, d_out_scores, stream=0):
        self._ck(self.L.oi_search_bm25_dev(self.h, _addr(d_terms), _addr(d_offs), nq, k, _addr(d_out_ids), _addr(d_out_scores), stream))

    def search_hybrid_dev(self, d_queries, d_terms, d_offs, nq, k, rrf_k, d_ids, d_rrf, d_rc, d_rb, stream=0):
        self._ck(self.L.oi_search_hybrid_dev(self.h, _addr(d_queries), _addr(d_terms), _addr(d_offs), nq, k, rrf_k,
                                             _addr(d_ids), _addr(d_rrf), _addr(d_rc), _addr(d_rb), stream))

    def debug_cosine_gemm_scores(self, queries):
        """tests: raw nq x n_docs score matrix of the tensor-core path"""
        queries = np.ascontiguousarray(queries, dtype=np.float32).reshape(-1, self.dim)
        out = np.empty((queries.shape[0], self.n_docs), dtype=np.float32)
        self._ck(self.L.oi_debug_cosine_gemm_scores(self.h, _addr(queries), queries.shape[0], _addr(out)))
        return out

    def launch_count(self):
        return int(self.L.oi_index_launch_count(self.h))

    def set_option(self, name, value):
        self._ck(self.L.oi_index_set_option(self.h, name.encode(), int(value)))


def summaries_from_array(a):
    """SOCIAL_SUMMARY_DTYPE array -> list of summary dicts shaped like GpuLexicon's"""
    return [{f: (int(r[f]) if t is C.c_uint64 else float(r[f])) for f, t in SocialSummary._fields_} for r in a]


def summaries_to_array(summaries):
    """list of summary dicts -> SOCIAL_SUMMARY_DTYPE array (the layout of oi_social_summary)"""
    out = np.zeros(len(summaries), dtype=SOCIAL_SUMMARY_DTYPE)
    for i, sm in enumerate(summaries):
        for f, _ in SocialSummary._fields_:
            out[i][f] = sm[f]
    return out


def pack_texts(texts):
    """list of str (encoded as UTF-8) or bytes -> (blob u8[], offsets u64[n + 1]) as the text entry points take them"""
    raw = [t.encode("utf-8") if isinstance(t, str) else bytes(t) for t in texts]
    offs = np.zeros(len(raw) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(r) for r in raw])
    blob = np.frombuffer(b"".join(raw) or b"\0", dtype=np.uint8).copy()
    return blob, offs


def unpack_terms(blob, offsets):
    """(bytes, offsets) of a vocabulary or of gathered vocabularies -> list of str"""
    raw = np.asarray(blob, dtype=np.uint8).tobytes()
    offs = np.asarray(offsets, dtype=np.int64)
    return [raw[offs[t]:offs[t + 1]].decode("ascii") for t in range(len(offs) - 1)]


class GpuLexicon:
    """The handle form of the GPU PostAnalyzer (oi_lexicon_*): stream and device buffers live as long as the object."""

    def __init__(self, device=0, reserve_bytes=1 << 20, reserve_posts=1 << 12):
        self.L = load_library()
        self.h = C.c_void_p()
        s = self.L.oi_lexicon_create(device, reserve_bytes, reserve_posts, C.byref(self.h))
        if s:
            self.h = None
            raise OiError(s, self.L.oi_last_error(None).decode())

    def close(self):
        if getattr(self, "h", None):
            self.L.oi_lexicon_destroy(self.h)
            self.h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def run_packed(self, blob, offs, summary=False, threshold=0.2):
        """(blob, offsets) from pack_texts -> (polarity f64[n], speculative bool[n], bull u32[n], bear u32[n][, summary dict])"""
        n = len(offs) - 1
        pol = np.empty(n, dtype=np.float64)
        spec = np.empty(n, dtype=np.uint8)
        bull = np.empty(n, dtype=np.uint32)
        bear = np.empty(n, dtype=np.uint32)
        sm = SocialSummary()
        s = self.L.oi_lexicon_run(self.h, _addr(blob), _addr(offs), n, _addr(pol), _addr(spec), _addr(bull), _addr(bear),
                                  threshold, C.byref(sm) if summary else None)
        if s:
            raise OiError(s, self.L.oi_last_error(None).decode())
        out = (pol, spec.astype(bool), bull, bear)
        if summary:
            out += ({f: getattr(sm, f) for f, _ in SocialSummary._fields_},)
        return out

    def analyze(self, texts, summary=False, threshold=0.2):
        return self.run_packed(*pack_texts(texts), summary=summary, threshold=threshold)

    def launch_count(self):
        return int(self.L.oi_lexicon_launch_count(self.h))


def lexicon_analyze(texts, device=0):
    """Batched GPU PostAnalyzer: list of str -> (polarity f64[n], speculative bool[n], bull u32[n], bear u32[n])."""
    L = load_library()
    raw = [t.encode("utf-8") for t in texts]
    offs = np.zeros(len(raw) + 1, dtype=np.uint64)
    offs[1:] = np.cumsum([len(r) for r in raw])
    blob = np.frombuffer(b"".join(raw) or b"\0", dtype=np.uint8).copy()
    n = len(raw)
    pol = np.empty(n, dtype=np.float64)
    spec = np.empty(n, dtype=np.uint8)
    bull = np.empty(n, dtype=np.uint32)
    bear = np.empty(n, dtype=np.uint32)
    s = L.oi_lexicon_analyze(device, _addr(blob), _addr(offs), n, _addr(pol), _addr(spec), _addr(bull), _addr(bear))
    if s:
        raise OiError(s, L.oi_last_error(None).decode())
    return pol, spec.astype(bool), bull, bear
