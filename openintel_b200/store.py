"""SQLite post store and the index builder that lifts a GPU hybrid index out of it
(SURVEY.md §8 row a5 and §8(f) rank 1; BASELINE.json configs[0] "SQLite-backed").

The reference keeps no store of any kind (SURVEY.md §0), so the schema is ours; it mirrors the
reference's document type field for field -- `SocialPost {id, source, author, text, created_at,
engagement}` (src/domain/entities/social_post.rs:30-38), `PostText::parse` (trimmed, non-empty,
at most 10 000 chars: social_post.rs:7-23), `SourceKind {Reddit, Bluesky}` rendered as
"reddit" / "bluesky" (src/domain/values/source_kind.rs:5-20) -- plus one embedding per post.

    store  --posts, in doc_id order-->  oi_index_build_bm25_text: the reference tokenizer (src/adapters/analyzer/
                                        lexicon.rs:54-58), vocabulary and CSR built on the device
           --embeddings (f32 BLOBs)-->  L2-normalise in f32 (SPEC §2)            -->  oi_index_load_embeddings

The document-sharded lift (lift_shard_gpu, ShardedStoreIndex) runs on the device too: every rank builds its doc range
with oi_index_build_bm25_text, the ranks all-gather their packed vocabularies, and oi_index_bm25_union_vocabulary forms
the sorted union and re-indexes the shard's lists to the global term ids.

lift_csr and lift_shard (host tokenizer + IndexBuilder, C++) build the same vocabularies and CSRs on the host: they are
the references the device builds are tested against.

Scoring happens in libopenintel_gpu.so only; nothing here computes a score.
"""
import datetime
import sqlite3

import numpy as np

from . import capi, fusion, hostlib

MAX_POST_LEN = 10_000  # chars, not bytes (social_post.rs:7, :19)
SOURCES = ("reddit", "bluesky")

SCHEMA = """
CREATE TABLE IF NOT EXISTS posts (
  doc_id     INTEGER PRIMARY KEY,                              -- dense row id 0..N-1 = the index's u32 doc id
  id         TEXT    NOT NULL UNIQUE,                          -- SocialPost.id
  source     TEXT    NOT NULL CHECK (source IN ('reddit', 'bluesky')),
  author     TEXT    NOT NULL,
  text       TEXT    NOT NULL,                                 -- PostText: trimmed, non-empty, <= 10 000 chars
  created_at TEXT    NOT NULL,                                 -- RFC 3339, UTC
  engagement INTEGER NOT NULL CHECK (engagement BETWEEN 0 AND 4294967295)
);
CREATE TABLE IF NOT EXISTS embeddings (
  doc_id INTEGER PRIMARY KEY REFERENCES posts(doc_id),
  vec    BLOB NOT NULL                                         -- dim x f32, little endian
);
CREATE TABLE IF NOT EXISTS meta (key TEXT PRIMARY KEY, value TEXT NOT NULL);
"""


class InvalidPostText(ValueError):
    """DomainError::InvalidPostText (src/domain/error.rs) for rows that PostText::parse would reject"""


# Rust's str::trim() strips the Unicode White_Space set; Python's bare str.strip() also strips U+001C..U+001F
_WHITE_SPACE = "\t\n\x0b\x0c\r \x85\xa0\u1680\u2000\u2001\u2002\u2003\u2004\u2005\u2006\u2007\u2008\u2009\u200a\u2028\u2029\u202f\u205f\u3000"


def _dedupe(ids):
    """first-seen-order de-duplication of a query's term ids (ADVICE r1: the 64-term limit counts distinct terms)"""
    return np.array(list(dict.fromkeys(int(t) for t in ids)), dtype=np.uint32)


def parse_post_text(raw):
    """PostText::parse (social_post.rs:13-23): Unicode-whitespace trim, reject empty and > 10 000 chars."""
    t = raw.strip(_WHITE_SPACE)
    if not t:
        raise InvalidPostText("empty")
    if len(t) > MAX_POST_LEN:
        raise InvalidPostText("exceeds max length")
    return t


_EPOCH = datetime.datetime(1970, 1, 1, tzinfo=datetime.timezone.utc)


def parse_created_at(text):
    """A post's creation time (SPEC §8b): RFC 3339 with a UTC offset ('Z' or +-HH:MM) -> whole seconds since the Unix
    epoch, fractional seconds floored.  A value without an offset is refused (ValueError): its instant is unknown."""
    dt = datetime.datetime.fromisoformat(text)
    if dt.utcoffset() is None:
        raise ValueError("created_at %r has no UTC offset" % (text,))
    d = dt - _EPOCH  # a timedelta keeps 0 <= seconds < 86400 and 0 <= microseconds: this is the floor
    return d.days * 86400 + d.seconds


def open_store(path=":memory:", dim=None):
    """Opens (creating if needed) a post store.  `dim` fixes the embedding dimension of a new store."""
    conn = sqlite3.connect(path)
    conn.executescript(SCHEMA)
    if dim is not None:
        cur = conn.execute("SELECT value FROM meta WHERE key = 'dim'").fetchone()
        if cur is None:
            conn.execute("INSERT INTO meta (key, value) VALUES ('dim', ?)", (str(int(dim)),))
        elif int(cur[0]) != int(dim):
            raise ValueError("store holds %s-dim embeddings, not %d" % (cur[0], dim))
    conn.commit()
    return conn


def store_dim(conn):
    cur = conn.execute("SELECT value FROM meta WHERE key = 'dim'").fetchone()
    return int(cur[0]) if cur else None


def insert_posts(conn, posts, embeddings=None):
    """Appends posts (dicts with the SocialPost fields) and, optionally, their embeddings [n][dim] f32.
    doc ids continue from the current row count so they stay dense.  Text is validated like PostText::parse."""
    n0 = conn.execute("SELECT COUNT(*) FROM posts").fetchone()[0]
    rows = []
    for i, p in enumerate(posts):
        if p["source"] not in SOURCES:
            raise ValueError("unknown source %r" % (p["source"],))
        rows.append((n0 + i, p["id"], p["source"], p["author"], parse_post_text(p["text"]), p["created_at"], int(p["engagement"])))
    emb, dim = None, store_dim(conn)
    if embeddings is not None:
        emb = np.ascontiguousarray(embeddings, dtype="<f4")
        if emb.ndim != 2 or emb.shape[0] != len(rows) or (dim is not None and emb.shape[1] != dim):
            raise ValueError("embeddings must be [%d][%s] f32" % (len(rows), dim))
    with conn:  # one transaction: a rejected batch leaves the store unchanged
        conn.executemany("INSERT INTO posts (doc_id, id, source, author, text, created_at, engagement) VALUES (?,?,?,?,?,?,?)", rows)
        if emb is not None:
            if dim is None:
                conn.execute("INSERT INTO meta (key, value) VALUES ('dim', ?)", (str(emb.shape[1]),))
            conn.executemany("INSERT INTO embeddings (doc_id, vec) VALUES (?, ?)", ((n0 + i, emb[i].tobytes()) for i in range(len(rows))))
    return n0, len(rows)


def iter_posts(conn, chunk=4096):
    """(doc_id, id, text) in doc_id order, `chunk` rows at a time"""
    cur = conn.execute("SELECT doc_id, id, text FROM posts ORDER BY doc_id")
    while True:
        rows = cur.fetchmany(chunk)
        if not rows:
            return
        yield rows


def normalise_rows_f32(rows):
    """SPEC §2: stored rows are L2-normalised at build time -- f32 sum of squares in index order is not
    required (any association), so numpy's f32 pairwise sum is fine; a zero row stays zero."""
    rows = np.ascontiguousarray(rows, dtype=np.float32)
    n = np.sqrt(np.einsum("ij,ij->i", rows, rows, dtype=np.float32)).astype(np.float32)
    n[n == 0] = 1.0
    return rows / n[:, None]


def to_bf16_rne(rows):
    """f32 -> bf16 bit patterns (uint16), round to nearest even (SPEC §2 bf16 path); finite inputs"""
    u = np.ascontiguousarray(rows, dtype=np.float32).view(np.uint32)
    return ((u + np.uint32(0x7FFF) + ((u >> np.uint32(16)) & np.uint32(1))) >> np.uint32(16)).astype(np.uint16)


def lift_csr(conn, chunk=4096):
    """Tokenises every post with the reference tokenizer and builds vocabulary + CSR on the host.
    -> (IndexBuilder, csr dict, post ids in doc order)"""
    b = hostlib.IndexBuilder()
    ids = []
    expect = 0
    for rows in iter_posts(conn, chunk):
        for doc_id, _, _ in rows:
            if doc_id != expect:
                raise ValueError("posts.doc_id must be dense 0..N-1 (gap at %d)" % expect)
            expect += 1
        ids.extend(r[1] for r in rows)
        b.add([r[2] for r in rows])
    csr = b.finish()
    return b, csr, ids


def lift_embeddings(conn, n_docs, dim, chunk=8192):
    """[n_docs][dim] f32, L2-normalised, in doc_id order; a post without an embedding is an error."""
    out = np.empty((n_docs, dim), dtype=np.float32)
    cur = conn.execute("SELECT doc_id, vec FROM embeddings ORDER BY doc_id")
    got = 0
    while True:
        rows = cur.fetchmany(chunk)
        if not rows:
            break
        for doc_id, blob in rows:
            if doc_id != got:
                raise ValueError("embedding missing for doc %d" % got)
            v = np.frombuffer(blob, dtype="<f4")
            if v.shape[0] != dim:
                raise ValueError("doc %d: embedding has %d components, store says %d" % (doc_id, v.shape[0], dim))
            out[got] = v
            got += 1
    if got != n_docs:
        raise ValueError("embedding missing for doc %d" % got)
    return normalise_rows_f32(out)


class Vocabulary:
    """The vocabulary of an index built from text on the device: term id i = terms[i] (ascending byte order).
    Maps query text to term ids with the rules of IndexBuilder.query_terms."""

    def __init__(self, terms):
        self.terms = terms
        self.ids = {w: i for i, w in enumerate(terms)}

    def term(self, term_id):
        return self.terms[term_id]

    def query_terms(self, text):
        """term ids of the text's tokens: unknown tokens dropped, duplicates dropped in first-seen order (SPEC §3)"""
        return _dedupe([self.ids[t] for t in hostlib.tokenize(text) if t in self.ids])

    def close(self):
        pass


class StoreIndex:
    """A GPU hybrid index built from a post store: the drop-in search side of the path.

    search(texts, vectors, k) tokenises the query texts with the same tokenizer as the documents, maps tokens
    to term ids (unknown tokens are dropped), normalises the query vectors and calls oi_search_hybrid."""

    def __init__(self, conn, dtype=capi.DTYPE_F32, device=0, max_k=100, max_batch=16, k1=1.2, b=0.75):
        self.conn = conn
        texts, self.post_ids = [], []
        for rows in iter_posts(conn):
            for doc_id, post_id, text in rows:
                if doc_id != len(texts):
                    raise ValueError("posts.doc_id must be dense 0..N-1 (gap at %d)" % len(texts))
                texts.append(text)
                self.post_ids.append(post_id)
        self.n_docs = len(texts)
        self.dim = store_dim(conn)
        if self.dim is None:
            raise ValueError("store has no embeddings")
        rows = lift_embeddings(conn, self.n_docs, self.dim)
        self.ix = capi.GpuIndex(n_docs=self.n_docs, dim=self.dim, dtype=dtype, device=device, max_k=max_k, max_batch=max_batch)
        try:
            # a bf16 index stores the normalised rows rounded to nearest even (SPEC §2)
            self.ix.load_embeddings(to_bf16_rne(rows) if dtype == capi.DTYPE_BF16 else rows)
            self.builder = Vocabulary(self.ix.build_bm25_text(texts))
            self.n_terms = self.ix.n_terms
            self.ix.bm25_finalize(k1=k1, b=b)
        except Exception:
            self.ix.close()
            raise

    def query_terms(self, texts):
        """term ids of each query text: unknown tokens dropped, duplicates dropped in first-seen order (SPEC §3)"""
        return [_dedupe(self.builder.query_terms(t)) for t in texts]

    def search(self, texts, vectors, k, rrf_k=60):
        q = normalise_rows_f32(np.asarray(vectors, dtype=np.float32).reshape(len(texts), self.dim))
        ids, rrf, rc, rb = self.ix.search_hybrid(q, self.query_terms(texts), k, rrf_k)
        hits = []
        for j in range(len(texts)):
            hits.append([dict(doc_id=int(d), id=self.post_ids[int(d)], rrf=float(s), rank_cosine=int(c), rank_bm25=int(bm))
                         for d, s, c, bm in zip(ids[j], rrf[j], rc[j], rb[j]) if d != capi.NO_DOC])
        return hits

    def close(self):
        self.ix.close()
        self.builder.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


# ---- document-sharded lift (one process per GPU, SPEC §5) ----------------------------------------
def lift_shard(conn, dist, rank=None, world=None, device="cpu"):
    """This rank's share of a document-sharded index, lifted out of the store every rank can read:

      * the rank tokenises ONLY its contiguous doc range (sharding.shard_range),
      * the vocabularies are unioned over the ranks (all_gather_object) so term ids are GLOBAL: the sorted union,
        i.e. exactly the ids the unsharded lift assigns,
      * the shard's CSR is re-indexed to the global vocabulary (absent terms = empty lists, doc ids shard-local),
      * df / doc-length sums are all-reduced (sharding.global_bm25_stats), so every shard scores with global
        N, avgdl and idf.

    `dist` = torch.distributed (initialised, gloo or nccl) or None.  -> dict(doc_base, n_local, n_docs_global, vocab,
    csr (global vocabulary), global_df, avgdl, post_ids (this shard's))"""
    from . import sharding
    n_total = conn.execute("SELECT COUNT(*) FROM posts").fetchone()[0]
    if dist is not None and dist.get_world_size() > 1:
        rank, world = dist.get_rank(), dist.get_world_size()
    else:
        dist, rank, world = None, 0, 1
    base, n_local = sharding.shard_range(n_total, world, rank)
    b = hostlib.IndexBuilder()
    ids = []
    cur = conn.execute("SELECT doc_id, id, text FROM posts WHERE doc_id >= ? AND doc_id < ? ORDER BY doc_id", (base, base + n_local))
    expect = base
    while True:
        rows = cur.fetchmany(4096)
        if not rows:
            break
        for doc_id, _, _ in rows:
            if doc_id != expect:
                raise ValueError("posts.doc_id must be dense 0..N-1 (gap at %d)" % expect)
            expect += 1
        ids.extend(r[1] for r in rows)
        b.add([r[2] for r in rows])
    if expect != base + n_local:
        raise ValueError("posts.doc_id must be dense 0..N-1 (gap at %d)" % expect)
    local = b.finish()
    local_vocab = [b.term(i) for i in range(local["n_terms"])]
    b.close()
    if dist is not None:
        gathered = [None] * world
        dist.all_gather_object(gathered, local_vocab)
        vocab = sorted(set().union(*gathered))
    else:
        vocab = local_vocab
    # local term id -> global term id (both lists are sorted, so the map is increasing)
    pos = {w: i for i, w in enumerate(vocab)}
    gid = np.array([pos[w] for w in local_vocab], dtype=np.int64)
    lens = np.zeros(len(vocab), dtype=np.uint64)
    if len(gid):
        lens[gid] = np.diff(local["term_offsets"])
    off = np.zeros(len(vocab) + 1, dtype=np.uint64)
    np.cumsum(lens, out=off[1:])
    csr = dict(term_offsets=off, doc_ids=local["doc_ids"], tfs=local["tfs"], doc_len=local["doc_len"],
               n_docs=n_local, n_terms=len(vocab))  # postings keep their order: lists are concatenated by term id
    gdf, avgdl, n = sharding.global_bm25_stats(dist, lens.astype(np.uint32), int(local["doc_len"].sum()), n_local, device=device)
    if n != n_total:
        raise ValueError("the ranks see %d posts in total, the store holds %d" % (n, n_total))
    return dict(doc_base=base, n_local=n_local, n_docs_global=n_total, vocab=vocab, csr=csr, global_df=gdf, avgdl=float(avgdl),
                post_ids=ids)


def lift_shard_gpu(conn, dist, device="cpu", device_index=0, max_k=100, max_batch=16, with_embeddings=True):
    """lift_shard on the device: the same shard, built into an open GpuIndex on `device_index` --
      * the rank's contiguous doc range is tokenised and indexed by oi_index_build_bm25_text,
      * the packed vocabularies are all-gathered (sharding.all_gather_packed) and oi_index_bm25_union_vocabulary
        forms their sorted union and re-indexes the shard's CSR to it (global term ids, absent terms = empty lists),
      * df / doc-length sums are all-reduced (sharding.global_bm25_stats).
    A shard whose posts hold no token contributes no vocabulary; it forms the union on the host from the gathered
    entries and loads an all-empty CSR over it.

    `dist` = torch.distributed (initialised, gloo or nccl) or None; `device` = where its collectives run.  The index is
    not finalized: load the embeddings, then bm25_finalize with global_df / avgdl / n_docs_global.  with_embeddings=False:
    an index for the BM25 part alone (mention summaries, SPEC §8a) -- the store needs no embeddings and the index holds
    the smallest row it takes (4 f32), never loaded.  -> dict(index, doc_base, n_local, n_docs_global, vocab, global_df,
    avgdl, post_ids (this shard's))"""
    from . import sharding
    n_total = conn.execute("SELECT COUNT(*) FROM posts").fetchone()[0]
    if dist is not None and dist.get_world_size() > 1:
        rank, world = dist.get_rank(), dist.get_world_size()
    else:
        dist, rank, world = None, 0, 1
    base, n_local = sharding.shard_range(n_total, world, rank)
    texts, ids = [], []
    cur = conn.execute("SELECT doc_id, id, text FROM posts WHERE doc_id >= ? AND doc_id < ? ORDER BY doc_id", (base, base + n_local))
    for doc_id, post_id, text in cur:
        if doc_id != base + len(texts):
            raise ValueError("posts.doc_id must be dense 0..N-1 (gap at %d)" % (base + len(texts)))
        texts.append(text)
        ids.append(post_id)
    if len(texts) != n_local:
        raise ValueError("posts.doc_id must be dense 0..N-1 (gap at %d)" % (base + len(texts)))
    dim = store_dim(conn) if with_embeddings else 4
    if dim is None:
        raise ValueError("store has no embeddings")
    ix = capi.GpuIndex(n_docs=n_local, dim=dim, device=device_index, doc_base=base, max_k=max_k, max_batch=max_batch)
    try:
        no_token = None
        try:
            ix.build_bm25_text(texts)
            blob, offs = ix.read_vocabulary_packed()
        except capi.OiError as e:
            if e.status != 1 or "no token" not in e.message:
                raise
            no_token, blob, offs = e, np.zeros(0, np.uint8), np.zeros(1, np.uint64)
        blob, offs = sharding.all_gather_packed(dist, blob, offs, device=device)
        if no_token is not None:
            vocab = sorted(set(capi.unpack_terms(blob, offs)))
            if not vocab:  # no rank holds a token: the store cannot be indexed, sharded or not
                raise no_token
            ix.load_bm25(np.zeros(len(vocab) + 1, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint32),
                         np.zeros(n_local, np.uint32))
        else:
            vocab = ix.bm25_union_vocabulary(blob, offs)
        df, sum_dl, _ = ix.bm25_local_stats()
        gdf, avgdl, n = sharding.global_bm25_stats(dist, df, sum_dl, n_local, device=device)
        if n != n_total:
            raise ValueError("the ranks see %d posts in total, the store holds %d" % (n, n_total))
    except Exception:
        ix.close()
        raise
    return dict(index=ix, doc_base=base, n_local=n_local, n_docs_global=n_total, vocab=vocab, global_df=gdf,
                avgdl=float(avgdl), post_ids=ids)


class ShardedStoreIndex:
    """StoreIndex over the GPUs of one box: every rank lifts its doc range on its GPU (lift_shard_gpu), loads its
    embeddings, finalizes with GLOBAL BM25 statistics and joins the NCCL communicator; search() returns the same global
    lists on every rank."""

    def __init__(self, conn, dist, device_index=0, max_k=100, max_batch=16, k1=1.2, b=0.75):
        from . import sharding
        self.dist = dist if (dist is not None and dist.get_world_size() > 1) else None
        dev = "cuda:%d" % device_index
        sh = lift_shard_gpu(conn, self.dist, device=dev if self.dist else "cpu", device_index=device_index, max_k=max_k,
                            max_batch=max_batch)
        self.ix = sh["index"]
        self.vocab, self.doc_base, self.n_local, self.n_docs = sh["vocab"], sh["doc_base"], sh["n_local"], sh["n_docs_global"]
        self.term_id = {w: i for i, w in enumerate(self.vocab)}
        self.dim = store_dim(conn)
        try:
            rows = np.empty((self.n_local, self.dim), dtype=np.float32)
            cur = conn.execute("SELECT doc_id, vec FROM embeddings WHERE doc_id >= ? AND doc_id < ? ORDER BY doc_id",
                               (self.doc_base, self.doc_base + self.n_local))
            got = 0
            for doc_id, blob in cur:
                if doc_id != self.doc_base + got:
                    raise ValueError("embedding missing for doc %d" % (self.doc_base + got))
                rows[got] = np.frombuffer(blob, dtype="<f4")
                got += 1
            if got != self.n_local:
                raise ValueError("embedding missing for doc %d" % (self.doc_base + got))
            self.ix.load_embeddings(normalise_rows_f32(rows))
            self.ix.bm25_finalize(k1=k1, b=b, avgdl=sh["avgdl"], n_docs_global=self.n_docs, global_df=sh["global_df"])
            if self.dist:
                self.ix.comm_init(self.dist.get_rank(), self.dist.get_world_size(), sharding.broadcast_unique_id(self.dist, device=dev))
        except Exception:
            self.ix.close()
            raise

    def query_terms(self, texts):
        return [_dedupe([self.term_id[t] for t in hostlib.tokenize(x) if t in self.term_id]) for x in texts]

    def search(self, texts, vectors, k, rrf_k=60):
        q = normalise_rows_f32(np.asarray(vectors, dtype=np.float32).reshape(len(texts), self.dim))
        return self.ix.search_hybrid(q, self.query_terms(texts), k, rrf_k)

    def close(self):
        self.ix.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def _mentions_by_source(state):
    """{source name: post count} of a mention state (capi.MENTION_STATE_DTYPE), {} for none"""
    return {} if state is None else {SOURCES[s]: int(state["by_source"][s]) for s in range(len(SOURCES))}


def _social_block(state, summary):
    """the "social" block (analyze.social_block) of a mention state and its summary; None, None: no post"""
    from . import analyze
    return analyze.social_block(analyze.empty_summary() if summary is None else summary, _mentions_by_source(state))


class MentionIndex:
    """Per-ticker social reports from the index (SPEC §8a): the posts that mention a ticker are its posting list, so
    the reference's `analyze --mention` report of many tickers takes one device call (one relay over the ranks of a
    document-sharded index) instead of a pass over the store per ticker.

    Every rank lifts its doc range through lift_shard_gpu (unsharded when `dist` is None; the store needs no
    embeddings), scores its posts with the GPU PostAnalyzer and loads the signals and source codes next to the BM25
    part.  reports() returns on every rank exactly what analyze.analyze_posts returns for select_posts(source,
    mention=ticker).  timeline() splits the same summaries by creation time (SPEC §8b); mention_counts() counts every
    term's mentions by creation time and trending() ranks the terms by the surge of their counts (SPEC §8c);
    comention_counts() counts every term's posts together with tickers in a window and related() ranks the terms by
    their excess over independence, with the social block of the shared posts (SPEC §8d); authors() groups the tickers'
    posts by author and measures how concentrated the talk is (SPEC §8e).  These read the post times (and authors() the
    post authors) from `conn` on their first call, so `conn` stays open while the index is used."""

    def __init__(self, conn, dist=None, device_index=0):
        self.dist = dist if (dist is not None and dist.get_world_size() > 1) else None
        # the relay's control plane: CPU tensors over gloo, the rank's GPU over NCCL
        self.device = "cpu" if self.dist is None or self.dist.get_backend() == "gloo" else "cuda:%d" % device_index
        sh = lift_shard_gpu(conn, self.dist, device=self.device, device_index=device_index, max_k=1, max_batch=1,
                            with_embeddings=False)
        self.ix = sh["index"]
        self.vocab = sh["vocab"]
        self.term_id = {w: i for i, w in enumerate(self.vocab)}
        self.doc_base, self.n_local = sh["doc_base"], sh["n_local"]
        self.conn, self.times_loaded, self.authors_loaded = conn, False, False
        try:
            rows = conn.execute("SELECT source, text FROM posts WHERE doc_id >= ? AND doc_id < ? ORDER BY doc_id",
                                (self.doc_base, self.doc_base + self.n_local)).fetchall()
            with capi.GpuLexicon(device_index) as lx:
                pol, spec, _, _ = lx.analyze([r[1] for r in rows])
            self.source_codes = np.array([SOURCES.index(r[0]) for r in rows], dtype=np.uint8)
            self.ix.load_post_signals(pol, spec, self.source_codes)
        except Exception:
            self.ix.close()
            raise

    def reports(self, tickers, source=None, markets=None, cfg=fusion.EngineConfig()):
        """one report per ticker, in the order given: analyze.build_report of the ticker's posts (of `source` only, when
        given).  A ticker is normalised like select_posts' mention (analyze.ticker_key); `markets` maps tickers,
        normalised the same way, to fusion.MarketSummary.  A ticker with no post and no market snapshot -- what analyze
        refuses with NoData -- gives None."""
        from . import analyze, sharding
        mk = {analyze.ticker_key(k): v for k, v in (markets or {}).items()}
        out = []
        for k, st, sm in self._relay(tickers, sharding.relay_mention_summary, source, cfg):
            try:
                out.append(analyze.build_report(analyze.empty_summary() if sm is None else sm, _mentions_by_source(st),
                                                mk.get(k), cfg))
            except analyze.NoData:
                out.append(None)
        return out

    @staticmethod
    def _source_code(source):
        """a source name (store.SOURCES) -> its code; None (all posts) stays None"""
        return None if source is None else SOURCES.index(source)

    def _relay(self, tickers, relay, source, cfg, *args):
        """`relay` (sharding.relay_mention_summary, or relay_mention_timeline with the edges in `args`) over the distinct
        tickers in the vocabulary, normalised by analyze.ticker_key.  -> per ticker, in the order given, (normalised
        ticker, states, summaries); (ticker, None, None) for one outside the vocabulary, which has no post"""
        from . import analyze
        keys = [analyze.ticker_key(t) for t in tickers]
        known = [k for k in dict.fromkeys(keys) if k in self.term_id]
        states, sums = relay(self.dist, self.ix, np.array([self.term_id[k] for k in known], dtype=np.uint32), *args,
                             self._source_code(source), cfg.bull_bear_threshold, device=self.device)
        found = dict(zip(known, zip(states, sums)))
        return [(k,) + found.get(k, (None, None)) for k in keys]

    def _load_times(self):
        """parses this shard's created_at and loads it next to the BM25 part.  Sharded, the ranks agree first on whether
        every rank parsed its rows, so a bad row on one rank raises on all of them instead of leaving the others waiting
        in the relay."""
        rows = self.conn.execute("SELECT doc_id, created_at FROM posts WHERE doc_id >= ? AND doc_id < ? ORDER BY doc_id",
                                 (self.doc_base, self.doc_base + self.n_local)).fetchall()
        err, times = None, np.zeros(len(rows), dtype=np.int64)
        for i, (doc_id, text) in enumerate(rows):
            try:
                times[i] = parse_created_at(text)
            except ValueError as e:
                err = "post doc_id %d: %s" % (doc_id, e)
                break
        if self.dist is not None:
            import torch
            bad = torch.tensor([0 if err is None else 1], dtype=torch.int64, device=self.device)
            self.dist.all_reduce(bad, op=self.dist.ReduceOp.SUM)
            if err is None and int(bad.item()):
                err = "created_at of another shard's post is not RFC 3339 with a UTC offset"
        if err is not None:
            raise ValueError(err)
        self.ix.load_post_times(times)
        self.times, self.times_loaded = times, True

    def _edges(self, edges):
        """the bucket edges as ints, checked; the post times are read from the store and loaded on the first call"""
        edges = [int(e) for e in edges]
        if len(edges) < 2 or any(a >= b for a, b in zip(edges, edges[1:])):
            raise ValueError("edges must be at least two strictly increasing times")
        if not self.times_loaded:
            self._load_times()
        return edges

    def timeline(self, tickers, edges, source=None, cfg=fusion.EngineConfig()):
        """per ticker, in the order given, a list of len(edges) - 1 "social" blocks (analyze.social_block): block b
        summarises the ticker's posts (of `source` only, when given) created in [edges[b], edges[b + 1]), seconds since
        the Unix epoch -- what analyze_posts(select_posts(source, mention=ticker, since=edges[b], until=edges[b + 1]))
        reports as "social".  Tickers are normalised like reports(); one outside the vocabulary gets empty blocks.  The
        post times are read from the store and loaded on the first call; sharded, every rank calls with the same
        arguments."""
        return self._timeline(tickers, self._edges(edges), source, cfg)

    def _timeline(self, tickers, edges, source, cfg):
        from . import sharding
        out = []
        for _, states, sums in self._relay(tickers, sharding.relay_mention_timeline, source, cfg, edges):
            pairs = zip(states, sums) if sums is not None else [(None, None)] * (len(edges) - 1)  # no post
            out.append([_social_block(st, sm) for st, sm in pairs])
        return out

    def mention_counts(self, edges, source=None):
        """count[t][b] = the number of posts (of `source` only, when given) that mention term t of the vocabulary and
        were created in [edges[b], edges[b + 1]), seconds since the Unix epoch (SPEC §8c): one device call per shard over
        all terms, and an all-reduce of the shards' counts.  The post times are read from the store and loaded on the
        first call; sharded, every rank calls with the same arguments.  -> int64 [len(vocab)][len(edges) - 1], the same
        on every rank"""
        from . import sharding
        counts = self.ix.mention_counts(self._edges(edges), self._source_code(source))
        return sharding.all_reduce_counts(self.dist, counts, device=self.device)

    def trending(self, since, until, baseline_since, k, min_mentions=1, source=None, universe=None, cfg=fusion.EngineConfig()):
        """the terms whose mentions in the window [since, until) rise most above what the baseline [baseline_since, since)
        predicts, ranked by SPEC §8c (trending.rank): at most k entries {ticker, mentions, baseline_mentions, expected,
        surge, social: {baseline, window}}, where the social blocks are those of timeline() over the two windows.  Only
        terms with at least min_mentions mentions in the window are ranked; `universe` (tickers, normalised like
        reports()) restricts the ranking to its entries, and one outside the vocabulary is never ranked.  Times are
        seconds since the Unix epoch; sharded, every rank calls with the same arguments and gets the same list."""
        from . import trending
        t0, t1, t2, k, min_mentions = trending.check_args(baseline_since, since, until, k, min_mentions)
        counts = self.mention_counts([t0, t1, t2], source)
        ids, expected, surge = trending.rank(counts[:, 1], counts[:, 0], t0, t1, t2, k, min_mentions,
                                             self._universe_mask(universe))
        blocks = self._timeline([self.vocab[t] for t in ids], [t0, t1, t2], source, cfg)
        return [{"ticker": self.vocab[t], "mentions": int(counts[t, 1]), "baseline_mentions": int(counts[t, 0]),
                 "expected": float(x), "surge": float(sg), "social": {"baseline": b[0], "window": b[1]}}
                for t, x, sg, b in zip(ids, expected, surge, blocks)]

    def _universe_mask(self, universe):
        """a bool mask over the vocabulary of the universe's entries, normalised like reports(); None for all terms.  An
        entry outside the vocabulary marks nothing."""
        from . import analyze
        if universe is None:
            return None
        mask = np.zeros(len(self.vocab), dtype=bool)
        mask[[self.term_id[w] for w in map(analyze.ticker_key, universe) if w in self.term_id]] = True
        return mask

    def _comention_batches(self, keys, window, source):
        """the co-mention counts of the normalised tickers `keys` (distinct, all in the vocabulary) against every term,
        in device calls of at most capi.MAX_COMENTION_ANCHORS anchors, all-reduced over the shards.  -> per batch,
        (its keys, int64 [len(keys)][len(vocab)])"""
        from . import sharding
        for i in range(0, len(keys), capi.MAX_COMENTION_ANCHORS):
            batch = keys[i:i + capi.MAX_COMENTION_ANCHORS]
            counts = self.ix.comention_counts([self.term_id[k] for k in batch], window, self._source_code(source))
            yield batch, sharding.all_reduce_counts(self.dist, counts, device=self.device)

    def comention_counts(self, tickers, since, until, source=None):
        """co[i][u] = the number of posts (of `source` only, when given) created in [since, until), seconds since the
        Unix epoch, that mention both tickers[i] and term u of the vocabulary (SPEC §8d): one device call per shard and
        batch of at most 64 distinct tickers, and an all-reduce of the shards' counts.  Tickers are normalised like
        reports(); one outside the vocabulary is never sent to the device and gets a row of zeros.  The post times are
        read from the store and loaded on the first call; sharded, every rank calls with the same arguments.
        -> int64 [len(tickers)][len(vocab)], the same on every rank"""
        from . import analyze
        window = self._edges([since, until])
        keys = [analyze.ticker_key(t) for t in tickers]
        rows = {}
        for batch, counts in self._comention_batches([k for k in dict.fromkeys(keys) if k in self.term_id], window, source):
            rows.update(zip(batch, counts))
        out = np.zeros((len(keys), len(self.vocab)), dtype=np.int64)
        for i, k in enumerate(keys):
            if k in rows:
                out[i] = rows[k]
        return out

    def _window_posts(self, since, until, source):
        """N of SPEC §8d: the posts (of `source` only, when given) created in [since, until), over all shards"""
        from . import sharding
        inside = (self.times >= since) & (self.times < until)
        if source is not None:
            inside &= self.source_codes == self._source_code(source)
        return int(sharding.all_reduce_counts(self.dist, np.array([np.count_nonzero(inside)]), device=self.device)[0])

    def related(self, tickers, since, until, k, min_co_mentions=1, source=None, universe=None, cfg=fusion.EngineConfig()):
        """per anchor ticker, in the order given, the terms mentioned together with it in the window [since, until)
        more often than independence predicts, ranked by SPEC §8d (related.rank): {ticker, mentions (n_a), posts (N),
        related: at most k entries {ticker, co_mentions, mentions (n_u), expected, score, social}}.  `social` is the
        "social" block of the posts in the window that mention both, so its total_mentions is co_mentions.  Only terms
        with at least min_co_mentions co-mentions are ranked; `universe` (tickers, normalised like reports()) restricts
        the ranking to its entries, and one outside the vocabulary is never ranked.  An anchor outside the vocabulary,
        or with no post in the window, ranks nothing.  Times are seconds since the Unix epoch; one device call per shard
        and batch of 64 anchors for the counts, one relay per batch for the social blocks; sharded, every rank calls
        with the same arguments and gets the same result."""
        from . import analyze, related, sharding
        since, until, k, min_co_mentions = related.check_args(since, until, k, min_co_mentions)
        n_u = self.mention_counts([since, until], source)[:, 0]
        n_posts = self._window_posts(since, until, source)
        mask = self._universe_mask(universe)
        keys = [analyze.ticker_key(t) for t in tickers]
        found = {}
        for batch, counts in self._comention_batches([t for t in dict.fromkeys(keys) if t in self.term_id], [since, until],
                                                     source):
            ranked = []
            for key, co in zip(batch, counts):
                a = self.term_id[key]
                ranked.append((key, co, int(co[a])) + related.rank(co, n_u, co[a], n_posts, a, k, min_co_mentions, mask))
            pairs = [(self.term_id[key], int(u)) for key, _, _, ids, _, _ in ranked for u in ids]
            states, sums = sharding.relay_comention_summary(
                self.dist, self.ix, np.array([p[0] for p in pairs], dtype=np.uint32),
                np.array([p[1] for p in pairs], dtype=np.uint32), [since, until], self._source_code(source),
                cfg.bull_bear_threshold, device=self.device)
            j = 0
            for key, co, n_a, ids, expected, score in ranked:
                found[key] = (n_a, [{"ticker": self.vocab[u], "co_mentions": int(co[u]), "mentions": int(n_u[u]),
                                     "expected": float(x), "score": float(sc),
                                     "social": _social_block(states[j + i], sums[j + i])}
                                    for i, (u, x, sc) in enumerate(zip(ids, expected, score))])
                j += len(ids)
        return [{"ticker": key, "mentions": found.get(key, (0, []))[0], "posts": n_posts, "related": found.get(key, (0, []))[1]}
                for key in keys]

    def _load_authors(self):
        """reads this shard's source, author and engagement, numbers the authors and loads the ids next to the BM25 part.
        An author is (source, name); the ids are global and dense in (source code, UTF-8 name) order (SPEC §8e), so
        sharded the ranks all-gather their sorted distinct authors, packed as one source byte + the name, and every rank
        numbers their sorted union."""
        from . import sharding
        rows = self.conn.execute("SELECT source, author, engagement FROM posts WHERE doc_id >= ? AND doc_id < ? ORDER BY doc_id",
                                 (self.doc_base, self.doc_base + self.n_local)).fetchall()
        keys = [bytes([SOURCES.index(src)]) + name.encode("utf-8") for src, name, _ in rows]
        mine = sorted(set(keys))
        if self.dist is not None:
            blob, offs = capi.pack_texts(mine)
            blob, offs = sharding.all_gather_packed(self.dist, blob[:int(offs[-1])], offs, device=self.device)
            raw, offs = blob.tobytes(), offs.astype(np.int64)
            mine = sorted({raw[offs[i]:offs[i + 1]] for i in range(len(offs) - 1)})
        ids = {key: i for i, key in enumerate(mine)}
        self.ix.load_post_authors(np.array([ids[key] for key in keys], dtype=np.uint32),
                                  np.array([r[2] for r in rows], dtype=np.uint32))
        self.author_keys = [(SOURCES[key[0]], key[1:].decode("utf-8")) for key in mine]
        self.authors_loaded = True

    def authors(self, tickers, since, until, k, source=None, cfg=fusion.EngineConfig()):
        """per ticker, in the order given, who posted about it in the window [since, until) (of `source` only, when
        given) and how concentrated that talk is (SPEC §8e): {ticker, mentions (P), authors (A), effective_authors, hhi,
        top_share, engagement, top: at most k entries {source, author, posts, bullish, bearish, neutral, speculative,
        engagement, first_at, last_at}}, ranked by posts, then engagement, descending, then author.  Tickers are
        normalised like reports(); one outside the vocabulary, or without a post in the window, gets zeros and no
        entry.  Times are seconds since the Unix epoch; one device call per shard for all tickers, and the shards' runs
        are gathered and merged; sharded, every rank calls with the same arguments and gets the same result."""
        from . import analyze, authors, sharding
        since, until, k = authors.check_args(since, until, k)
        window = self._edges([since, until])
        if not self.authors_loaded:
            self._load_authors()
        keys = [analyze.ticker_key(t) for t in tickers]
        known = [t for t in dict.fromkeys(keys) if t in self.term_id]
        _, runs = self.ix.mention_authors(np.array([self.term_id[t] for t in known], dtype=np.uint32), window,
                                          self._source_code(source), cfg.bull_bear_threshold)
        if self.dist is not None:
            runs = authors.merge(sharding.all_gather_runs(self.dist, runs, device=self.device))
        cut = np.searchsorted(runs["term"], np.arange(len(known) + 1))
        found = {}
        for i, key in enumerate(known):
            r = authors.rank(runs[cut[i]:cut[i + 1]], k)
            top = [{"source": self.author_keys[int(x["author"])][0], "author": self.author_keys[int(x["author"])][1],
                    "posts": int(x["posts"]), "bullish": int(x["bullish"]), "bearish": int(x["bearish"]),
                    "neutral": int(x["posts"]) - int(x["bullish"]) - int(x["bearish"]), "speculative": int(x["speculative"]),
                    "engagement": int(x["engagement"]), "first_at": int(x["first_at"]), "last_at": int(x["last_at"])}
                   for x in r["top"]]
            found[key] = {"mentions": r["mentions"], "authors": r["authors"], "effective_authors": r["effective_authors"],
                          "hhi": r["hhi"], "top_share": r["top_share"], "engagement": r["engagement"], "top": top}
        none = {"mentions": 0, "authors": 0, "effective_authors": 0.0, "hhi": 0.0, "top_share": 0.0, "engagement": 0, "top": []}
        return [dict({"ticker": key}, **found.get(key, none)) for key in keys]

    def close(self):
        self.ix.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
