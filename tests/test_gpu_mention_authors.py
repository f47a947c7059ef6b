"""oi_index_mention_authors and the layers on top (SPEC §8e): the (term, author) runs of the posts in a window must equal
select_posts(mention, since, until) grouped by (source, author) on the host, unsharded and merged over the shards of a
document-sharded index; store.MentionIndex.authors must give the §8e figures and order; and the `authors` CLI must print
what MentionIndex.authors returns."""
import json
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from mention_util import G, oi  # noqa: F401  (fixtures)
from mention_util import (DAY, ROOT, T0, fixture_store, iso, make_store, run_ranks, sharded_corpus, small_corpus,
                          synthetic as _synthetic)

pytestmark = pytest.mark.gpu

SOURCES = (None, "reddit", "bluesky")
FIELDS = ("posts", "bullish", "bearish", "speculative", "engagement", "first_at", "last_at")


def author_store(path, texts, sources, authors, times, engagement):
    """a store without embeddings whose posts have the given authors and engagement"""
    from openintel_b200 import store
    conn = store.open_store(path)
    store.insert_posts(conn, [dict(id="p%d" % i, source=s, author=a, text=t, created_at=iso(tm), engagement=int(e))
                              for i, (t, s, a, tm, e) in enumerate(zip(texts, sources, authors, times, engagement))])
    return conn


def _author_order(key):
    """SPEC §8e author order: (source code, UTF-8 name)"""
    from openintel_b200 import store
    return store.SOURCES.index(key[0]), key[1].encode("utf-8")


class HostRuns:
    """the host oracle: every post's source, author, created_at, engagement and oracle lexicon scores, read back from the
    store; the runs of a ticker are its posts grouped by (source, author)"""

    def __init__(self, conn):
        from openintel_b200 import store
        rows = conn.execute("SELECT id, source, author, text, created_at, engagement FROM posts ORDER BY doc_id").fetchall()
        self.rows = rows
        self.index = {r[0]: d for d, r in enumerate(rows)}
        self.times = np.array([store.parse_created_at(r[4]) for r in rows], dtype=np.int64)
        scores = [O.lexicon_score(r[3]) for r in rows]
        self.pol = np.array([s[0] for s in scores])
        self.spec = np.array([s[1] for s in scores], dtype=np.int64)
        self.src = np.array([r[1] for r in rows])
        self.eng = np.array([r[5] for r in rows], dtype=np.int64)
        self.keys = sorted({(r[1], r[2]) for r in rows}, key=_author_order)
        kid = {k: i for i, k in enumerate(self.keys)}
        self.author = np.array([kid[(r[1], r[2])] for r in rows], dtype=np.int64)
        self._posting = None

    def group(self, docs, thr):
        """[(source, author, posts, bullish, bearish, speculative, engagement, first_at, last_at)] of the posts `docs`,
        in SPEC §8e author order"""
        docs = np.asarray(docs, dtype=np.int64)
        ids, inv = np.unique(self.author[docs], return_inverse=True)
        n = len(ids)
        lo, hi = np.full(n, np.iinfo(np.int64).max), np.full(n, np.iinfo(np.int64).min)
        np.minimum.at(lo, inv, self.times[docs])
        np.maximum.at(hi, inv, self.times[docs])
        eng = np.zeros(n, dtype=np.int64)
        np.add.at(eng, inv, self.eng[docs])

        def count(flag):
            return np.bincount(inv, weights=flag.astype(np.int64), minlength=n).astype(np.int64)
        cols = (np.bincount(inv, minlength=n), count(self.pol[docs] > thr), count(self.pol[docs] < -thr),
                count(self.spec[docs]), eng, lo, hi)
        return [self.keys[a] + tuple(int(c[j]) for c in cols) for j, a in enumerate(ids)]

    def select(self, conn, ticker, window, source, thr=0.2):
        """the runs of select_posts(source, mention=ticker, since, until)"""
        from openintel_b200 import analyze
        ids = analyze.select_posts(conn, source=source, mention=ticker, since=window[0], until=window[1])[0]
        return self.group([self.index[i] for i in ids], thr)

    def runs(self, vocab, term, window, source, thr=0.2):
        """the same from one tokenisation of the corpus (for the large corpus: one pass instead of one per ticker)"""
        from openintel_b200 import hostlib
        if self._posting is None:
            self._posting = {}
            for d, r in enumerate(self.rows):
                for w in set(hostlib.tokenize(r[3])):
                    self._posting.setdefault(w, []).append(d)
        docs = np.array(self._posting.get(vocab[term], []), dtype=np.int64)
        keep = (self.times[docs] >= window[0]) & (self.times[docs] < window[1])
        if source is not None:
            keep &= self.src[docs] == source
        return self.group(docs[keep], thr)


def device_runs(mi, term_ids, window, source, thr=0.2, capacity=4096):
    """the raw call through MentionIndex's author ids -> per term index, [(source, author, fields...)] in run order"""
    from openintel_b200 import store
    if not mi.authors_loaded:
        mi.authors(["x"], window[0], window[1], 1)  # loads the times and the authors
    code = None if source is None else store.SOURCES.index(source)
    term_runs, runs = mi.ix.mention_authors(np.array(term_ids, dtype=np.uint32), window, code, thr, capacity=capacity)
    assert term_runs.dtype == np.uint64 and len(term_runs) == len(term_ids) + 1 and int(term_runs[-1]) == len(runs)
    assert (runs["term"] == np.repeat(np.arange(len(term_ids)), np.diff(term_runs.astype(np.int64)))).all()
    out = []
    for i in range(len(term_ids)):
        r = runs[int(term_runs[i]):int(term_runs[i + 1])]
        assert (np.diff(r["author"].astype(np.int64)) > 0).all()  # ascending author id: (source, name) order
        out.append([mi.author_keys[int(x["author"])] + tuple(int(x[f]) for f in FIELDS) for x in r])
    return out


def _check_invariants(mi, term_ids, window, source, thr=0.2):
    """P = the §8c count; the class sums = the one-bucket timeline state"""
    from openintel_b200 import store
    code = None if source is None else store.SOURCES.index(source)
    got = device_runs(mi, term_ids, window, source, thr)
    counts = mi.ix.mention_counts(window, code)[:, 0]
    states, _ = mi.ix.mention_timeline(np.array(term_ids, dtype=np.uint32), window, code, thr)
    for i, t in enumerate(term_ids):
        assert sum(r[2] for r in got[i]) == int(counts[t]) == int(states[i, 0]["total"])
        for j, f in ((3, "bullish"), (4, "bearish"), (5, "speculative")):
            assert sum(r[j] for r in got[i]) == int(states[i, 0][f]), (t, f)
    return got


# ---- 1. runs against the host oracle ----------------------------------------------------------------------------------
def test_fixture_runs_equal_select_posts(oi, G, tmp_path):
    from openintel_b200 import store
    conn, _, hours = fixture_store(G, str(tmp_path / "fixture.db"))
    n = len(hours)
    on = T0 + 3600 * int(np.sort(hours)[3])  # a post exactly on since, and one exactly on until (left out)
    with store.MentionIndex(conn) as mi:
        host = HostRuns(conn)
        words = ["aapl", "calls", "the", "puts", "aapl"]  # a duplicate term
        ids = [mi.term_id[w] for w in words]
        for w in ([T0, T0 + 3600 * n], [on, on + 3600 * 4], [T0 - 3600 * 5, T0]):
            for src in SOURCES:
                for thr in (0.2, 0.05):
                    got = _check_invariants(mi, ids, w, src, thr)
                    for word, g in zip(words, got):
                        assert g == host.select(conn, word, w, src, thr), (word, w, src, thr)
        assert got[0] == got[4]
    conn.close()


def test_small_corpus_runs(oi, tmp_path):
    from openintel_b200 import store
    texts, _, _, src, times = small_corpus()
    conn = make_store(str(tmp_path / "small.db"), texts, [store.SOURCES[s] for s in src], times)
    with store.MentionIndex(conn) as mi:
        host = HostRuns(conn)
        for w in ([T0, T0 + 51 * 3600], [T0 + 10 * 3600, T0 + 40 * 3600], [T0 + 60 * 3600, T0 + 70 * 3600]):
            for s in SOURCES:
                got = _check_invariants(mi, [mi.term_id[x] for x in ("gme", "amc", "puts")], w, s)
                assert got == [host.select(conn, x, w, s) for x in ("gme", "amc", "puts")]
        # gme: posts 0 (a0, reddit, hour 50), 1 (a1, bluesky, hour 10) and 4 (a4, bluesky, hour 40, "GME GME": once)
        got = device_runs(mi, [mi.term_id["gme"]], [T0, T0 + 51 * 3600], None)[0]
        assert [(r[0], r[1], r[2], r[7]) for r in got] == [("reddit", "a0", 1, T0 + 50 * 3600), ("bluesky", "a1", 1, T0 + 10 * 3600),
                                                         ("bluesky", "a4", 1, T0 + 40 * 3600)]
    conn.close()


N_SYN = 200_000


@pytest.fixture(scope="module")
def synthetic(oi, tmp_path_factory):
    from openintel_b200 import store
    texts, sources, tickers = _synthetic(N_SYN, 2027)
    rng = np.random.default_rng(81)
    times = T0 + rng.integers(0, 60 * DAY, N_SYN)
    times[rng.random(N_SYN) < 0.05] = T0 + 20 * DAY  # posts exactly on a window's since
    times[rng.random(N_SYN) < 0.05] = T0 + 30 * DAY  # ... and on its until
    conn = make_store(str(tmp_path_factory.mktemp("authors") / "syn.db"), texts, sources, times)
    mi = store.MentionIndex(conn)
    yield dict(conn=conn, mi=mi, host=HostRuns(conn), tickers=tickers)
    mi.close()
    conn.close()


SYN_WINDOWS = {"all": [T0 - DAY, T0 + 61 * DAY], "edges": [T0 + 20 * DAY, T0 + 30 * DAY], "none": [T0 - 9 * DAY, T0 - DAY]}


@pytest.mark.parametrize("window", sorted(SYN_WINDOWS))
@pytest.mark.parametrize("n_terms", [1, 64, 1000])
def test_synthetic_runs_equal_the_host_oracle(oi, synthetic, window, n_terms):
    S = synthetic
    mi, host = S["mi"], S["host"]
    known = [t for t in S["tickers"] if t in mi.term_id]
    words = known + ["calls", "the", "moon"]
    ids = [mi.term_id[words[i % len(words)]] for i in range(n_terms)]  # 1000 ids hold duplicates
    w = SYN_WINDOWS[window]
    for src in SOURCES:
        got = _check_invariants(mi, ids, w, src)
        want = {}
        for i, t in enumerate(ids):
            if t not in want:
                want[t] = host.runs(mi.vocab, t, w, src)
            assert got[i] == want[t], (window, src, mi.vocab[t])
        if window == "none":
            assert not any(got)
    if n_terms == 64 and window == "edges":  # the head ticker through select_posts itself
        for src in SOURCES:
            assert device_runs(mi, [ids[0]], w, src)[0] == host.select(S["conn"], known[0], w, src)
        # authors post on both sources: (reddit, a5) and (bluesky, a5) are two authors
        names = [r[:2] for r in device_runs(mi, [ids[0]], w, None)[0]]
        assert ("reddit", "a5") in names and ("bluesky", "a5") in names


def test_synthetic_capacity_refusal(oi, synthetic):
    from openintel_b200 import capi
    mi = synthetic["mi"]
    device_runs(mi, [0], SYN_WINDOWS["all"], None)
    ids = np.array([mi.term_id[t] for t in synthetic["tickers"][:5] if t in mi.term_id], dtype=np.uint32)
    w = np.array(SYN_WINDOWS["all"], dtype=np.int64)
    want_tr, want = mi.ix.mention_authors(ids, w, capacity=1)  # refused once, then retried at the reported count
    need = len(want)
    assert need > 100
    tr = np.full(len(ids) + 1, 7, dtype=np.uint64)
    runs = np.zeros(need, dtype=capi.AUTHOR_RUN_DTYPE)
    runs["posts"] = 9
    import ctypes as C
    n = C.c_uint64(0)
    for cap in (0, need - 1):
        s = mi.ix.L.oi_index_mention_authors(mi.ix.h, ids.ctypes.data, len(ids), w.ctypes.data, -1, 0.2, cap, tr.ctypes.data,
                                             runs.ctypes.data, C.byref(n))
        assert s == 1 and n.value == need and "capacity" in mi.ix.L.oi_last_error(mi.ix.h).decode()
        assert (tr == 7).all() and (runs["posts"] == 9).all() and not runs["author"].any()  # nothing else written
    s = mi.ix.L.oi_index_mention_authors(mi.ix.h, ids.ctypes.data, len(ids), w.ctypes.data, -1, 0.2, need, tr.ctypes.data,
                                         runs.ctypes.data, C.byref(n))
    assert s == 0 and n.value == need and (tr == want_tr).all() and runs.tobytes() == want.tobytes()
    tr2, again = mi.ix.mention_authors(ids, w, capacity=need + 1000)
    assert (tr2 == want_tr).all() and again.tobytes() == want.tobytes()


# ---- 2. errors and state ------------------------------------------------------------------------------------------------
def _raw(ix, terms, n, window, source=-1, capacity=64, tr=None, runs=None, n_out=None):
    from openintel_b200 import capi
    return ix.L.oi_index_mention_authors(ix.h, capi._addr(terms), n, capi._addr(window), source, 0.2, capacity,
                                         capi._addr(tr), capi._addr(runs), n_out)


@pytest.mark.parametrize("loaded", [(), ("bm25",), ("bm25", "signals"), ("bm25", "signals", "times"),
                                    ("bm25", "signals", "authors"), ("signals", "times", "authors")])
def test_a_call_before_its_data_is_refused(oi, loaded):
    import ctypes as C
    from openintel_b200 import capi
    texts, pol, spec, src, times = small_corpus()
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        if "bm25" in loaded:
            ix.build_bm25_text(texts)
        if "signals" in loaded:
            ix.load_post_signals(pol, spec, src)
        if "times" in loaded:
            ix.load_post_times(times)
        if "authors" in loaded:
            ix.load_post_authors(np.arange(len(texts)), np.ones(len(texts)))
        n = C.c_uint64(0)
        tr, runs = np.zeros(2, np.uint64), np.zeros(4, dtype=capi.AUTHOR_RUN_DTYPE)
        assert _raw(ix, np.zeros(1, np.uint32), 1, np.array([T0, T0 + DAY], np.int64), tr=tr, runs=runs, n_out=C.byref(n)) == 5
        missing = ("BM25" if "bm25" not in loaded else "signals" if "signals" not in loaded else
                   "times" if "times" not in loaded else "authors")
        assert missing in ix.L.oi_last_error(ix.h).decode()


def test_errors_and_state(oi):
    import ctypes as C
    from openintel_b200 import capi
    texts, pol, spec, src, times = small_corpus()
    w = np.array([T0, T0 + 51 * 3600], dtype=np.int64)
    author = np.array([2, 0, 2, 1, 0, 2], dtype=np.uint32)
    eng = np.array([5, 6, 7, 8, 9, 2 ** 32 - 1], dtype=np.uint32)
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        vocab = ix.build_bm25_text(texts)
        V = len(vocab)
        ix.load_post_signals(pol, spec, src)
        ix.load_post_times(times)
        gme, amc = vocab.index("gme"), vocab.index("amc")
        with pytest.raises(capi.OiError) as e:
            ix.mention_authors([gme], w)
        assert e.value.status == 5 and "oi_index_load_post_authors" in e.value.message
        with pytest.raises(capi.OiError) as e:  # NULL author: refused
            ix._ck(ix.L.oi_index_load_post_authors(ix.h, None, capi._addr(eng)))
        assert e.value.status == 1
        ix.load_post_authors(author, eng)
        tr0, r0 = ix.mention_authors([gme, amc, gme], w)
        # gme: posts 0 (author 2), 1 (author 0), 4 (author 0); amc: posts 2 (author 2), 5 (author 2)
        assert tr0.tolist() == [0, 2, 3, 5] and r0["author"].tolist() == [0, 2, 2, 0, 2]
        assert r0["posts"].tolist() == [2, 1, 2, 2, 1] and r0["engagement"].tolist() == [15, 5, 7 + 2 ** 32 - 1, 15, 5]
        assert r0["first_at"].tolist()[:3] == [T0 + 10 * 3600, T0 + 50 * 3600, T0] and r0["last_at"][0] == T0 + 40 * 3600
        dup = r0[3:].copy()
        dup["term"] = 0
        assert r0["term"].tolist() == [0, 0, 1, 2, 2] and dup.tobytes() == r0[:2].tobytes()  # a duplicate term
        # refusals: each one writes nothing, and the next call gives the same runs
        bad = [dict(terms=None), dict(window=None), dict(tr=None), dict(runs=None), dict(n_out=None),
               dict(window=np.array([T0, T0], dtype=np.int64)), dict(window=np.array([T0 + 5, T0], dtype=np.int64)),
               dict(source=2), dict(source=-2), dict(terms=np.array([gme, V], dtype=np.uint32))]
        for kw in bad:
            n = C.c_uint64(77)
            args = dict(terms=np.array([gme, amc], dtype=np.uint32), window=w, tr=np.full(3, 7, np.uint64),
                        runs=np.zeros(8, dtype=capi.AUTHOR_RUN_DTYPE), n_out=C.byref(n))
            args.update(kw)
            assert _raw(ix, args["terms"], 2, args["window"], kw.get("source", -1), 8, args["tr"], args["runs"], args["n_out"]) == 1, kw
            assert n.value == 77 and (args["tr"] is None or (args["tr"] == 7).all()), kw
            assert args["runs"] is None or not args["runs"].view(np.uint8).any(), kw
            tr, r = ix.mention_authors([gme, amc, gme], w)
            assert (tr == tr0).all() and r.tobytes() == r0.tobytes(), kw
        # zero terms: a no-op, with any pointers
        assert _raw(ix, None, 0, None, 9, 0, None, None, None) == 0
        tr, r = ix.mention_authors([], w)
        assert tr.tolist() == [0] and len(r) == 0
        # a window without a post: no run
        tr, r = ix.mention_authors([gme, amc], [T0 - DAY, T0])
        assert tr.tolist() == [0, 0, 0] and len(r) == 0
        # before and after finalize, a rebuilt BM25 part and reloaded signals keep the authors
        ix.bm25_finalize()
        assert ix.mention_authors([gme, amc, gme], w)[1].tobytes() == r0.tobytes()
        assert ix.build_bm25_text(texts) == vocab
        ix.load_post_signals(pol, spec, src)
        assert ix.mention_authors([gme, amc, gme], w)[1].tobytes() == r0.tobytes()
        # a refused load keeps the previous authors; new ones replace them
        assert ix.L.oi_index_load_post_authors(ix.h, capi._addr(author), None) == 1
        assert ix.mention_authors([gme, amc, gme], w)[1].tobytes() == r0.tobytes()
        ix.load_post_authors(np.full(6, 2 ** 32 - 1, np.uint32), eng)  # the widest key: n_authors = 2^32
        tr, r = ix.mention_authors([gme, amc, gme], w)
        assert tr.tolist() == [0, 1, 2, 3] and r["author"].tolist() == [2 ** 32 - 1] * 3 and r["posts"].tolist() == [3, 2, 3]
    # a shard without a posting: no run
    with oi.GpuIndex(n_docs=3, dim=4, max_k=1) as ix:
        ix.load_bm25(np.zeros(5, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(3, np.uint32))
        ix.load_post_signals(np.zeros(3), np.zeros(3, np.uint8), np.zeros(3, np.uint8))
        ix.load_post_times(np.full(3, T0, dtype=np.int64))
        ix.load_post_authors(np.arange(3), np.zeros(3))
        tr, r = ix.mention_authors([1, 3], w)
        assert tr.tolist() == [0, 0, 0] and len(r) == 0


# ---- 3. the sharded index over gloo ranks (all on device 0) ------------------------------------------------------------
W_SHARD = [T0 + DAY, T0 + 7 * DAY]
A_SHARD = ["onlyfirst", "$CALLS", "moon", "nope", "the"]


def _sharded_result(mi, head):
    return {str(src): json.dumps(mi.authors(A_SHARD + [head], W_SHARD[0], W_SHARD[1], 12, source=src)) for src in SOURCES}


def _sharded_worker(dist, path, head):
    from openintel_b200 import store
    conn = store.open_store(path)
    with store.MentionIndex(conn, dist) as mi:
        out = _sharded_result(mi, head)
    conn.close()
    return out


@pytest.mark.parametrize("world,tokenless", [(2, False), (3, False), (3, True)])
def test_sharded_authors_equal_the_unsharded_ones(oi, tmp_path, world, tokenless):
    from openintel_b200 import sharding, store
    texts, sources, tickers = sharded_corpus(41 + world, world, tokenless)
    times = T0 + np.random.default_rng(world + 9).integers(0, 8 * DAY, len(texts))
    times[[3, 10]] = T0 + 2 * DAY  # both onlyfirst posts in the window
    path = str(tmp_path / "posts.db")
    make_store(path, texts, sources, times).close()  # authors a{i % 97}: every author posts on every shard
    conn = store.open_store(path)
    with store.MentionIndex(conn) as mi:
        want = _sharded_result(mi, tickers[0])
        got = mi.authors([tickers[0]], *W_SHARD, 200)[0]  # the head ticker: most authors hold a run
        assert got["authors"] > 100 and got["mentions"] > got["authors"]
    conn.close()
    for r in range(world):
        base, n = sharding.shard_range(len(texts), world, r)
        if not (tokenless and r == 1):
            assert len({i % 97 for i in range(base, base + n)}) == 97
    for rank, got in run_ranks(world, _sharded_worker, path, tickers[0]):
        assert got == want, rank


# ---- 4. a planted corpus ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def planted(oi, tmp_path_factory):
    """one account with 500 posts on $SPAM, 500 accounts with one post each on $CROWD, and background talk"""
    rng = np.random.default_rng(7)
    texts, sources, authors, times, eng = [], [], [], [], []

    def post(text, source, author, t, e):
        texts.append(text)
        sources.append(source)
        authors.append(author)
        times.append(t)
        eng.append(e)
    for i in range(500):
        post("$SPAM to the moon %d" % i, "reddit", "spammer", T0 + DAY + 60 * i, 3)
    for i in range(500):
        post("$CROWD looks %s" % ("great buy" if i % 2 else "like a dump"), ("reddit", "bluesky")[i % 2], "user%03d" % i,
             T0 + DAY + 97 * i, i)
    for i in range(2000):
        post("background chatter %d the" % i, ("reddit", "bluesky")[i % 2], "bg%d" % (i % 40), T0 + int(rng.integers(0, 3 * DAY)),
             int(rng.integers(0, 100)))
    order = rng.permutation(len(texts))  # interleaved in doc order
    path = str(tmp_path_factory.mktemp("planted") / "planted.db")
    conn = author_store(path, [texts[i] for i in order], [sources[i] for i in order], [authors[i] for i in order],
                        [times[i] for i in order], [eng[i] for i in order])
    from openintel_b200 import store
    mi = store.MentionIndex(conn)
    yield dict(conn=conn, path=path, mi=mi)
    mi.close()
    conn.close()


def test_planted_concentration(oi, planted):
    mi = planted["mi"]
    spam, crowd, none = mi.authors(["$SPAM", "crowd", "notaword"], T0, T0 + 3 * DAY, 5)
    assert spam["ticker"] == "spam" and spam["mentions"] == 500 and spam["authors"] == 1
    assert (spam["hhi"], spam["effective_authors"], spam["top_share"]) == (1.0, 1.0, 1.0)
    assert spam["top"] == [{"source": "reddit", "author": "spammer", "posts": 500, "bullish": 500, "bearish": 0, "neutral": 0,
                            "speculative": 0, "engagement": 1500, "first_at": T0 + DAY, "last_at": T0 + DAY + 60 * 499}]
    assert spam["engagement"] == 1500
    assert crowd["mentions"] == 500 and crowd["authors"] == 500 and crowd["effective_authors"] == 500.0
    assert crowd["hhi"] == 1 / 500 and crowd["top_share"] == 5 / 500 and crowd["engagement"] == sum(range(500))
    # all tied on one post: engagement descending
    assert [(t["author"], t["engagement"]) for t in crowd["top"]] == [("user%03d" % i, i) for i in (499, 498, 497, 496, 495)]
    assert none == {"ticker": "notaword", "mentions": 0, "authors": 0, "effective_authors": 0.0, "hhi": 0.0, "top_share": 0.0,
                    "engagement": 0, "top": []}
    # a window that cuts the spammer's run, and a source filter
    cut = mi.authors(["spam"], T0 + DAY + 60 * 100, T0 + DAY + 60 * 200, 5)[0]
    assert cut["mentions"] == 100 and cut["top"][0]["first_at"] == T0 + DAY + 60 * 100
    assert mi.authors(["spam"], T0, T0 + 3 * DAY, 5, source="bluesky")[0]["mentions"] == 0
    blue = mi.authors(["crowd"], T0, T0 + 3 * DAY, 500, source="bluesky")[0]
    assert blue["authors"] == 250 and all(t["source"] == "bluesky" for t in blue["top"]) and blue["top_share"] == 1.0
    # "the": the spammer's 500 posts and the 2000 background posts of 40 accounts
    both = mi.authors(["the"], T0, T0 + 3 * DAY, 3)[0]
    assert both["mentions"] == 2000 + 500 and both["authors"] == 40 + 1
    with pytest.raises(ValueError):
        mi.authors(["spam"], T0, T0, 5)
    with pytest.raises(ValueError):
        mi.authors(["spam"], T0, T0 + DAY, 0)


# ---- 5. the authors CLI prints what MentionIndex.authors returns --------------------------------------------------------
def _cli(*args):
    return subprocess.run([sys.executable, "-m", "openintel_b200.authors"] + list(args), cwd=ROOT, capture_output=True,
                          text=True, timeout=300)


def test_authors_cli(oi, planted, tmp_path):
    from openintel_b200 import timeline
    since, until = T0, T0 + 3 * DAY
    t = [timeline.format_time(x) for x in (since, until)]
    mi = planted["mi"]
    want = json.loads(json.dumps(mi.authors(["$SPAM", "crowd"], since, until, 10)))
    want_src = json.loads(json.dumps(mi.authors(["crowd"], since, until, 3, source="reddit")))
    r = _cli("--store", planted["path"], "--since", t[0], "--until", t[1], "$SPAM", "crowd")
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout) == {"since": t[0], "until": t[1], "source": None, "top": 10, "tickers": want}
    r = _cli("--store", planted["path"], "--since", t[0], "--until", t[1], "--top", "3", "--source", "reddit", "crowd")
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["tickers"] == want_src
    bad = make_store(str(tmp_path / "bad.db"), ["gme moon"], ["reddit"], [T0])
    bad.execute("UPDATE posts SET created_at = '2024-01-01 00:00:00'")
    bad.commit()
    bad.close()
    r = _cli("--store", str(tmp_path / "bad.db"), "--since", t[0], "--until", t[1], "gme")
    assert r.returncode == 1 and r.stderr.startswith("error:") and "doc_id 0" in r.stderr
    assert _cli("--store", planted["path"], "--since", t[1], "--until", t[1], "gme").returncode == 2
