"""oi_index_comention_counts / oi_index_comention_summary and the layers on top (SPEC §8d): the co-mention counts of
anchors against every term must equal a host count over the tokenized posts, unsharded and summed over the shards of a
document-sharded index; the shared-post summaries must equal `analyze` over the posts that mention both terms, bit for
bit; and store.MentionIndex.related and the `related` CLI must rank the terms by the §8d rule."""
import json
import math
import subprocess
import sys

import numpy as np
import pytest

from mention_util import G, oi  # noqa: F401  (fixtures)
from mention_util import (DAY, ROOT, T0, bits as _bits, fixture_store, make_store, run_ranks, same_summary, sharded_corpus,
                          small_corpus, synthetic as _synthetic)

pytestmark = pytest.mark.gpu

SOURCES = (None, "reddit", "bluesky")


class HostCo:
    """the host oracle: per post, the set of its tokens (hostlib.tokenize), its source and its created_at
    (store.parse_created_at), read back from the store"""

    def __init__(self, conn, vocab):
        from openintel_b200 import hostlib, store
        rows = conn.execute("SELECT source, text, created_at FROM posts ORDER BY doc_id").fetchall()
        tid = {w: i for i, w in enumerate(vocab)}
        docs, terms = [], []
        for d, (_, text, _) in enumerate(rows):
            for w in set(hostlib.tokenize(text)):
                docs.append(d)
                terms.append(tid[w])
        self.docs, self.terms = np.array(docs, dtype=np.int64), np.array(terms, dtype=np.int64)
        self.src = np.array([r[0] for r in rows])
        self.times = np.array([store.parse_created_at(r[2]) for r in rows], dtype=np.int64)
        self.n_terms = len(vocab)

    def inside(self, window, source=None):
        """bool per post: in [since, until) and of the source"""
        keep = (self.times >= window[0]) & (self.times < window[1])
        if source is not None:
            keep &= self.src == source
        return keep

    def posts_of(self, term, window, source=None):
        """bool per post: mentions the term, in the window and of the source"""
        has = np.zeros(len(self.times), dtype=bool)
        has[self.docs[self.terms == term]] = True
        return has & self.inside(window, source)

    def co(self, anchor, window, source=None):
        """co(anchor, u) for every term u"""
        sel = self.posts_of(anchor, window, source)
        return np.bincount(self.terms[sel[self.docs]], minlength=self.n_terms).astype(np.int64)

    def counts(self, window, source=None):
        """every term's mention count in the window"""
        sel = self.inside(window, source)
        return np.bincount(self.terms[sel[self.docs]], minlength=self.n_terms).astype(np.int64)


def _check_counts(mi, oracle, anchors, window):
    """MentionIndex.comention_counts and the raw call against the oracle, for every source; co(a, a) = mention_counts
    and co(a, u) = co(u, a) over the anchors"""
    from openintel_b200 import store
    ids = [mi.term_id[a] for a in anchors]
    for src in SOURCES:
        code = None if src is None else store.SOURCES.index(src)
        got = mi.comention_counts(anchors, window[0], window[1], src)  # loads the post times on the first call
        assert got.dtype == np.int64 and got.shape == (len(anchors), len(mi.vocab))
        raw = mi.ix.comention_counts(ids, window, code)
        assert raw.dtype == np.uint32 and (raw == got).all()
        for i, a in enumerate(ids):
            assert (got[i] == oracle.co(a, window, src)).all(), (window, src, anchors[i])
        n_u = mi.mention_counts(window, src)[:, 0]
        assert (got[np.arange(len(ids)), ids] == n_u[ids]).all()  # co(a, a)
        assert (got[:, ids] == got[:, ids].T).all()  # co(a, u) == co(u, a)


# ---- 1. counts against the host oracle ------------------------------------------------------------------------------
def test_fixture_comention_counts_equal_the_host_oracle(oi, G, tmp_path):
    from openintel_b200 import store
    conn, _, hours = fixture_store(G, str(tmp_path / "fixture.db"))
    n = len(hours)
    on = T0 + 3600 * int(np.sort(hours)[3])  # a post exactly on since, and one exactly on until (left out)
    windows = [[T0, T0 + 3600 * n], [T0 + 3600 * 20 * n, T0 + 3600 * 21 * n], [on, on + 3600 * 4]]
    with store.MentionIndex(conn) as mi:
        oracle = HostCo(conn, mi.vocab)
        anchors = ["aapl", "calls", "the", "aapl"]  # a duplicate anchor gives an identical row
        for w in windows:
            _check_counts(mi, oracle, anchors, w)
        got = mi.comention_counts(["$AAPL", "calls", "zzzz", "AAPL"], *windows[0])
        assert (got[0] == got[3]).all() and not got[2].any() and int(got[0, mi.term_id["aapl"]]) == 10
        assert not mi.comention_counts(["aapl"], *windows[1]).any()
        inside = oracle.inside(windows[2])
        assert inside[oracle.times == on].all() and not inside[oracle.times == on + 3600 * 4].any()
    conn.close()


def test_small_corpus_comention_counts(oi, tmp_path):
    from openintel_b200 import store
    texts, _, _, src, times = small_corpus()
    conn = make_store(str(tmp_path / "small.db"), texts, [store.SOURCES[s] for s in src], times)
    with store.MentionIndex(conn) as mi:
        oracle = HostCo(conn, mi.vocab)
        for w in ([T0, T0 + 51 * 3600], [T0 + 10 * 3600, T0 + 40 * 3600], [T0 + 60 * 3600, T0 + 70 * 3600]):
            _check_counts(mi, oracle, ["gme", "amc", "puts", "gme"], w)
        # gme: posts 0 (hour 50), 1 (hour 10, "puts") and 4 (hour 40, "GME GME dump": counts once)
        c = mi.comention_counts(["gme"], T0, T0 + 51 * 3600)[0]
        assert [int(c[mi.term_id[w]]) for w in ("gme", "puts", "dump", "moon", "amc")] == [3, 1, 1, 1, 0]
    conn.close()


N_SYN = 200_000


@pytest.fixture(scope="module")
def synthetic(oi, tmp_path_factory):
    from openintel_b200 import store
    texts, sources, tickers = _synthetic(N_SYN, 2026)
    rng = np.random.default_rng(79)
    times = T0 + rng.integers(0, 60 * DAY, N_SYN)
    times[rng.random(N_SYN) < 0.05] = T0 + 20 * DAY  # posts exactly on a window's since
    times[rng.random(N_SYN) < 0.05] = T0 + 30 * DAY  # ... and on its until
    conn = make_store(str(tmp_path_factory.mktemp("comention") / "syn.db"), texts, sources, times)
    mi = store.MentionIndex(conn)
    yield dict(conn=conn, mi=mi, oracle=HostCo(conn, mi.vocab), tickers=tickers)
    mi.close()
    conn.close()


SYN_WINDOWS = {"all": [T0 - DAY, T0 + 61 * DAY], "edges": [T0 + 20 * DAY, T0 + 30 * DAY], "none": [T0 - 9 * DAY, T0 - DAY]}


@pytest.mark.parametrize("window", sorted(SYN_WINDOWS))
@pytest.mark.parametrize("n_anchors", [1, 63, 64])
def test_synthetic_comention_counts_equal_the_host_oracle(oi, synthetic, window, n_anchors):
    S = synthetic
    mi = S["mi"]
    known = [t for t in S["tickers"] if t in mi.term_id]
    anchors = ([known[0]] + known[1:n_anchors - 3] + ["calls", "the", known[0]])[:n_anchors]  # the head ticker, a duplicate
    assert len(anchors) == n_anchors
    _check_counts(mi, S["oracle"], anchors, SYN_WINDOWS[window])
    if window == "none":
        assert not mi.comention_counts(anchors, *SYN_WINDOWS[window]).any()


def test_synthetic_more_than_64_tickers_are_batched(oi, synthetic):
    S = synthetic
    mi = S["mi"]
    known = [t for t in S["tickers"] if t in mi.term_id][:70]
    w = SYN_WINDOWS["edges"]
    got = mi.comention_counts(known + ["$" + known[0].upper(), "notaword"], *w)
    assert got.shape == (72, len(mi.vocab)) and (got[70] == got[0]).all() and not got[71].any()
    for i in (0, 63, 64, 69):
        assert (got[i] == S["oracle"].co(mi.term_id[known[i]], w)).all()


# ---- 2. pair summaries against the host path -------------------------------------------------------------------------
def _host_pair(lx, conn, a, u, window, src, thr=0.2, cache=None):
    """(summary dict, {source: count}) of `analyze` over select_posts(mention=a, since, until) that also mention u;
    `cache` keeps select_posts' result per (a, window, source)"""
    from openintel_b200 import analyze, hostlib
    cache = {} if cache is None else cache
    key = (a, tuple(window), src)
    if key not in cache:
        cache[key] = analyze.select_posts(conn, source=src, mention=a, since=window[0], until=window[1])[1:]
    s, t = cache[key]
    keep = [i for i, x in enumerate(t) if u in hostlib.tokenize(x)]
    s, t = [s[i] for i in keep], [t[i] for i in keep]
    sm = lx.analyze(t, summary=True, threshold=thr)[4] if t else analyze.empty_summary()
    return sm, {x: s.count(x) for x in set(s)}


def _check_pairs(mi, conn, lx, anchors, terms, window, thresholds=(0.2, 0.05)):
    from openintel_b200 import analyze, store
    cache = {}
    a_ids = np.array([mi.term_id[a] for a in anchors], dtype=np.uint32)
    u_ids = np.array([mi.term_id[u] for u in terms], dtype=np.uint32)
    mi.mention_counts(window)  # loads the post times
    for src in SOURCES:
        code = None if src is None else store.SOURCES.index(src)
        co = mi.ix.comention_counts(np.unique(a_ids), window, code)
        row = {int(a): co[i] for i, a in enumerate(np.unique(a_ids))}
        for thr in thresholds:
            states, sums = mi.ix.comention_summary(a_ids, u_ids, window, code, thr)
            for j, (a, u) in enumerate(zip(anchors, terms)):
                want, by_src = _host_pair(lx, conn, a, u, window, src, thr, cache)
                same_summary(sums[j], want, (a, u, src, thr))
                assert int(states[j]["total"]) == int(row[int(a_ids[j])][u_ids[j]]) == want["total"]
                assert json.dumps(analyze.social_block(sums[j], store._mentions_by_source(states[j]))) == \
                    json.dumps(analyze.social_block(want, by_src))
            # pair(a, a) == the one-bucket timeline of a, bit for bit
            ts, tm = mi.ix.mention_timeline(a_ids, window, code, thr)
            ss, sm = mi.ix.comention_summary(a_ids, a_ids, window, code, thr)
            assert ss.tobytes() == ts[:, 0].tobytes()
            for x, y in zip(sm, tm):
                same_summary(x, y[0])


def test_fixture_pair_summaries_equal_analyze(oi, G, tmp_path):
    from openintel_b200 import capi, store
    conn, _, hours = fixture_store(G, str(tmp_path / "fixture.db"))
    n = len(hours)
    with capi.GpuLexicon() as lx, store.MentionIndex(conn) as mi:
        words = ["aapl", "calls", "the", "puts", "moon"]
        anchors = [a for a in words for _ in words]
        terms = [u for _ in words for u in words]
        for w in ([T0, T0 + 3600 * n], [T0 + 3600 * 2, T0 + 3600 * 9], [T0 - 3600 * 5, T0]):
            _check_pairs(mi, conn, lx, anchors, terms, w)
    conn.close()


def test_synthetic_pair_summaries_equal_analyze(oi, synthetic):
    from openintel_b200 import capi
    S = synthetic
    mi = S["mi"]
    known = [t for t in S["tickers"] if t in mi.term_id]
    anchors = [known[0], known[0], known[0], known[3], known[3], "calls", known[0]]
    terms = [known[1], "calls", known[0], known[0], "the", known[3], known[1]]  # a duplicate pair
    with capi.GpuLexicon() as lx:
        _check_pairs(mi, S["conn"], lx, anchors, terms, SYN_WINDOWS["edges"], thresholds=(0.2,))


# ---- 3. the sharded index over gloo ranks (all on device 0) ----------------------------------------------------------
W_SHARD = [T0 + DAY, T0 + 7 * DAY]
A_SHARD = ["onlyfirst", "$CALLS", "moon", "nope"]


def _sharded_result(mi):
    from openintel_b200 import sharding, store
    out = {}
    for src in SOURCES:
        out["counts", src] = mi.comention_counts(A_SHARD, W_SHARD[0], W_SHARD[1], src).tolist()
        out["related", src] = json.dumps(mi.related(A_SHARD, W_SHARD[0], W_SHARD[1], 12, source=src))
        ids = [mi.term_id[w] for w in ("onlyfirst", "calls", "moon")]
        st, sm = sharding.relay_comention_summary(mi.dist, mi.ix, np.repeat(ids, 3), np.tile(ids, 3), W_SHARD,
                                                  None if src is None else store.SOURCES.index(src), 0.2, device=mi.device)
        out["pairs", src] = (st.tobytes().hex(), json.dumps(sm))
    out["universe"] = json.dumps(mi.related(A_SHARD, W_SHARD[0], W_SHARD[1], 5, universe=["onlyfirst", "$MOON", "the", "nope"]))
    return {str(k): v for k, v in out.items()}


def _sharded_worker(dist, path):
    from openintel_b200 import store
    conn = store.open_store(path)
    with store.MentionIndex(conn, dist) as mi:
        out = _sharded_result(mi)
    conn.close()
    return out


@pytest.mark.parametrize("world,tokenless", [(2, False), (3, False), (3, True)])
def test_sharded_comentions_equal_the_unsharded_ones(oi, tmp_path, world, tokenless):
    from openintel_b200 import store
    texts, sources, _ = sharded_corpus(31 + world, world, tokenless)
    times = T0 + np.random.default_rng(world + 5).integers(0, 8 * DAY, len(texts))
    times[[3, 10]] = T0 + 2 * DAY  # both onlyfirst posts in the window
    path = str(tmp_path / "posts.db")
    make_store(path, texts, sources, times).close()
    conn = store.open_store(path)
    with store.MentionIndex(conn) as mi:
        want = _sharded_result(mi)
        c = mi.comention_counts(["onlyfirst"], *W_SHARD)[0]
        assert int(c[mi.term_id["onlyfirst"]]) == 2 and int(c[mi.term_id["moon"]]) >= 1 and int(c[mi.term_id["dump"]]) >= 1
    conn.close()
    for rank, got in run_ranks(world, _sharded_worker, path):
        assert got == want, rank


# ---- 4. related over a planted corpus ---------------------------------------------------------------------------------
TW, TE = T0 + 5 * DAY, T0 + 6 * DAY


def _rule(co, n_u, n_a, n_posts, anchor, k, min_co, allowed=None):
    """SPEC §8d in plain Python floats: [(term id, co, n_u, expected, score)] in rank order"""
    if n_a == 0:
        return []
    rows = []
    for u in range(len(co)):
        if u != anchor and co[u] >= min_co and (allowed is None or u in allowed):
            e = (float(int(n_a)) * float(int(n_u[u]))) / float(int(n_posts))
            rows.append((u, int(co[u]), int(n_u[u]), e, (float(int(co[u])) - e) / math.sqrt(e + 1.0)))
    rows.sort(key=lambda r: (-r[4], r[0]))
    return rows[:k]


@pytest.fixture(scope="module")
def planted(oi, tmp_path_factory):
    from openintel_b200 import store
    n = 8000
    texts, sources, tickers = _synthetic(n, 41, n_tickers=80)
    rng = np.random.default_rng(42)
    times = T0 + rng.integers(0, 10 * DAY, n)
    window = np.flatnonzero((times >= TW) & (times < TE))
    anchor_posts = rng.choice(window, size=len(window) // 3, replace=False)
    for i in anchor_posts:
        texts[i] += " $ANCH"
        if rng.random() < 0.9:
            texts[i] += " buddy"  # the partner: in most of the anchor's posts and nowhere else
    for i in range(n):
        if rng.random() < 0.5:
            texts[i] += " commonword"  # independent of the anchor
    path = str(tmp_path_factory.mktemp("related") / "planted.db")
    conn = make_store(path, texts, sources, times)
    mi = store.MentionIndex(conn)
    yield dict(conn=conn, path=path, mi=mi, oracle=HostCo(conn, mi.vocab), tickers=tickers)
    mi.close()
    conn.close()


@pytest.mark.parametrize("src", SOURCES)
def test_related_over_a_planted_corpus(oi, planted, src):
    from openintel_b200 import capi
    P = planted
    mi, O = P["mi"], P["oracle"]
    anchors = ["$ANCH", P["tickers"][0], "commonword", "notaword", "anch"]
    n_u = O.counts([TW, TE], src)
    n_posts = int(O.inside([TW, TE], src).sum())
    for k, mc in ((10, 1), (25, 3), (len(mi.vocab) + 5, 1), (5, 10 ** 6)):
        got = mi.related(anchors, TW, TE, k, min_co_mentions=mc, source=src)
        assert [g["ticker"] for g in got] == ["anch", P["tickers"][0], "commonword", "notaword", "anch"]
        assert got[0] == got[4] and got[3] == {"ticker": "notaword", "mentions": 0, "posts": n_posts, "related": []}
        for g in got[:3]:
            a = mi.term_id[g["ticker"]]
            co = O.co(a, [TW, TE], src)
            assert g["mentions"] == int(co[a]) and g["posts"] == n_posts
            want = _rule(co, n_u, co[a], n_posts, a, k, mc)
            assert [(mi.term_id[e["ticker"]], e["co_mentions"], e["mentions"], _bits(e["expected"]), _bits(e["score"]))
                    for e in g["related"]] == [(u, c, m, _bits(x), _bits(s)) for u, c, m, x, s in want], (g["ticker"], k, mc)
            assert all(e["social"]["total_mentions"] == e["co_mentions"] for e in g["related"])
    got = mi.related(["anch"], TW, TE, 10, source=src)[0]["related"]
    assert got[0]["ticker"] == "buddy"
    common = mi.related(["anch"], TW, TE, len(mi.vocab), source=src)[0]["related"]
    common = [e for e in common if e["ticker"] == "commonword"][0]
    assert abs(common["score"]) < 4.0 and common["co_mentions"] > 20
    # the social blocks are those of analyze over the shared posts
    with capi.GpuLexicon() as lx:
        from openintel_b200 import analyze
        for e in got[:4]:
            sm, by_src = _host_pair(lx, P["conn"], "anch", e["ticker"], [TW, TE], src)
            assert json.dumps(e["social"]) == json.dumps(analyze.social_block(sm, by_src))
    # a universe: normalised like --mention; entries outside the vocabulary are never ranked
    a = mi.term_id["anch"]
    co = O.co(a, [TW, TE], src)
    uni = ["BUDDY", "$commonword", "the", "$notaword", "anch"]
    allowed = {mi.term_id[w] for w in ("buddy", "commonword", "the", "anch")}
    got = mi.related(["anch"], TW, TE, 10, source=src, universe=uni)[0]["related"]
    assert [(e["ticker"], _bits(e["score"])) for e in got] == \
        [(mi.vocab[u], _bits(s)) for u, _, _, _, s in _rule(co, n_u, co[a], n_posts, a, 10, 1, allowed)]
    assert mi.related(["anch"], TW, TE, 10, source=src, universe=[])[0]["related"] == []
    # a window without a post
    assert mi.related(["anch"], T0 - 9 * DAY, T0 - DAY, 10, source=src) == \
        [{"ticker": "anch", "mentions": 0, "posts": 0, "related": []}]


def test_related_refuses_bad_arguments(oi, planted):
    mi = planted["mi"]
    for args in ((TW, TW, 5), (TE, TW, 5), (TW, TE, 0)):
        with pytest.raises(ValueError):
            mi.related(["anch"], *args)
    with pytest.raises(ValueError):
        mi.related(["anch"], TW, TE, 5, min_co_mentions=0)
    with pytest.raises(ValueError):
        mi.comention_counts(["anch"], TE, TW)


# ---- 5. errors and state ----------------------------------------------------------------------------------------------
def _raw_counts(ix, anchors, n, window, source=-1, out=None):
    from openintel_b200 import capi
    return ix.L.oi_index_comention_counts(ix.h, capi._addr(anchors), n, capi._addr(window), source, capi._addr(out))


def _raw_pairs(ix, a, u, n, window, source=-1, out=None, states=None):
    from openintel_b200 import capi
    return ix.L.oi_index_comention_summary(ix.h, capi._addr(a), capi._addr(u), n, capi._addr(window), source, 0.2, None,
                                           capi._addr(states), capi._addr(out))


def test_a_call_before_its_data_is_refused(oi):
    from openintel_b200 import capi
    texts, pol, spec, src, times = small_corpus()
    a = np.zeros(1, dtype=np.uint32)
    w = np.array([T0, T0 + DAY], dtype=np.int64)
    out = np.zeros(64, dtype=np.uint32)
    sums = np.zeros(1, dtype=capi.SOCIAL_SUMMARY_DTYPE)
    for load in ((), ("signals", "times"), ("bm25",), ("bm25", "signals"), ("bm25", "times")):
        with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
            if "bm25" in load:
                ix.build_bm25_text(texts)
            if "signals" in load:
                ix.load_post_signals(pol, spec, src)
            if "times" in load:
                ix.load_post_times(times)
            assert _raw_counts(ix, a, 1, w, out=out) == 5, load
            assert _raw_pairs(ix, a, a, 1, w, out=sums) == 5, load
            assert ("BM25" if "bm25" not in load else "signals" if "signals" not in load else "times") in \
                ix.L.oi_last_error(ix.h).decode()


def test_errors_and_state(oi):
    from openintel_b200 import capi
    texts, pol, spec, src, times = small_corpus()
    w = np.array([T0, T0 + 51 * 3600], dtype=np.int64)
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        vocab = ix.build_bm25_text(texts)
        V = len(vocab)
        ix.load_post_signals(pol, spec, src)
        ix.load_post_times(times)
        gme, amc, puts = vocab.index("gme"), vocab.index("amc"), vocab.index("puts")
        anchors = np.array([gme, amc], dtype=np.uint32)
        c0 = ix.comention_counts(anchors, w)
        assert c0.shape == (2, V) and c0[0, gme] == 3 and c0[0, puts] == 1 and c0[1, amc] == 2 and c0[1, gme] == 0
        pa, pu = np.array([gme, gme, amc], dtype=np.uint32), np.array([puts, gme, amc], dtype=np.uint32)
        s0, m0 = ix.comention_summary(pa, pu, w)
        assert [int(x) for x in s0["total"]] == [1, 3, 2]
        # refusals: each one writes nothing, and the next calls give the same results
        bad_counts = [dict(anchors=None), dict(window=None), dict(out=None), dict(window=np.array([T0, T0], dtype=np.int64)),
                      dict(window=np.array([T0 + 5, T0], dtype=np.int64)), dict(source=2), dict(source=-2),
                      dict(anchors=np.array([gme, V], dtype=np.uint32)), dict(n=65, anchors=np.full(65, gme, dtype=np.uint32))]
        for kw in bad_counts:
            n = kw.pop("n", 2)
            args = dict(anchors=anchors, window=w, out=np.full((n, V), 7, dtype=np.uint32))
            args.update(kw)
            out = args["out"]
            assert _raw_counts(ix, args["anchors"], n, args["window"], kw.get("source", -1), out) == 1, kw
            assert out is None or (out == 7).all(), kw
            assert (ix.comention_counts(anchors, w) == c0).all(), kw
        # 65 distinct anchor terms need a vocabulary that holds them
        with oi.GpuIndex(n_docs=2, dim=4, max_k=1) as big:
            bv = big.build_bm25_text([" ".join("w%d" % i for i in range(70)), "w0 w1"])
            big.load_post_signals(np.zeros(2), np.zeros(2, np.uint8), np.zeros(2, np.uint8))
            big.load_post_times(np.array([T0, T0 + 1], dtype=np.int64))
            ids = np.array([bv.index("w%d" % i) for i in range(65)], dtype=np.uint32)
            sums = np.zeros(65, dtype=capi.SOCIAL_SUMMARY_DTYPE)
            assert _raw_pairs(big, ids, ids, 65, w, out=sums) == 1 and not sums.view(np.uint8).any()
            st, sm = big.comention_summary(ids[:64], ids[::-1][:64], w)  # 64 distinct anchors are accepted
            assert [int(x) for x in st["total"]] == [1] * 64
            assert _raw_counts(big, ids, 65, w, out=np.zeros((65, len(bv)), np.uint32)) == 1
            assert big.comention_counts(ids[:64], w)[:, ids[0]].tolist() == [2, 2] + [1] * 62
        bad_pairs = [dict(a=None), dict(u=None), dict(window=None), dict(out=None), dict(window=np.array([T0, T0], dtype=np.int64)),
                     dict(source=2), dict(a=np.array([gme, V, amc], dtype=np.uint32)), dict(u=np.array([gme, gme, V], dtype=np.uint32))]
        for kw in bad_pairs:
            args = dict(a=pa, u=pu, window=w, out=np.zeros(3, dtype=capi.SOCIAL_SUMMARY_DTYPE))
            args.update(kw)
            out = args["out"]
            assert _raw_pairs(ix, args["a"], args["u"], 3, args["window"], kw.get("source", -1), out) == 1, kw
            assert out is None or not out.view(np.uint8).any(), kw
            s1, m1 = ix.comention_summary(pa, pu, w)
            assert s1.tobytes() == s0.tobytes() and m1 == m0, kw
        # zero anchors or pairs: a no-op, with any pointers
        out = np.full((1, V), 7, dtype=np.uint32)
        assert _raw_counts(ix, None, 0, None, 9, out) == 0 and (out == 7).all()
        assert _raw_pairs(ix, None, None, 0, None, 9, None) == 0
        assert ix.comention_counts([], w).shape == (0, V)
        # duplicates give identical rows; a larger call in between changes nothing
        d = ix.comention_counts([gme, amc, gme], w)
        assert (d[0] == d[2]).all() and (d[:2] == c0).all()
        assert ix.mention_counts(T0 - DAY + 3600 * np.arange(24 * 30 + 1, dtype=np.int64)).shape == (V, 24 * 30)
        assert (ix.comention_counts(anchors, w) == c0).all()
        # before and after finalize, a rebuilt BM25 part and reloaded signals: the same results
        ix.bm25_finalize()
        assert (ix.comention_counts(anchors, w) == c0).all()
        assert ix.build_bm25_text(texts) == vocab
        ix.load_post_signals(pol, spec, src)
        assert (ix.comention_counts(anchors, w) == c0).all()
        s1, m1 = ix.comention_summary(pa, pu, w)
        assert s1.tobytes() == s0.tobytes() and m1 == m0
        # a carry continues the states: the pair states plus a hand-made carry
        carry = np.zeros(3, dtype=capi.MENTION_STATE_DTYPE)
        carry["total"], carry["by_source"][:, 1] = 5, 5
        s2, _ = ix.comention_summary(pa, pu, w, carry=carry)
        assert (s2["total"] == s0["total"] + 5).all() and (s2["by_source"][:, 1] == s0["by_source"][:, 1] + 5).all()
        # new times move the posts out of the window
        ix.load_post_times(times + 60 * 3600)
        assert not ix.comention_counts(anchors, w).any()
    # a shard without a posting: zero counts and the carried states
    with oi.GpuIndex(n_docs=3, dim=4, max_k=1) as ix:
        ix.load_bm25(np.zeros(5, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(3, np.uint32))
        ix.load_post_signals(np.zeros(3), np.zeros(3, np.uint8), np.zeros(3, np.uint8))
        ix.load_post_times(np.full(3, T0, dtype=np.int64))
        out = np.full((2, 4), 7, dtype=np.uint32)
        assert _raw_counts(ix, np.array([1, 3], dtype=np.uint32), 2, w, out=out) == 0 and not out.any()
        carry = np.zeros(2, dtype=capi.MENTION_STATE_DTYPE)
        carry["total"], carry["sum"] = 4, 0.5
        st, sm = ix.comention_summary([1, 3], [2, 2], w, carry=carry)
        assert st.tobytes() == carry.tobytes() and [m["total"] for m in sm] == [4, 4]


# ---- 6. the related CLI prints what MentionIndex.related returns ----------------------------------------------------
def _cli(*args):
    return subprocess.run([sys.executable, "-m", "openintel_b200.related"] + list(args), cwd=ROOT, capture_output=True,
                          text=True, timeout=300)


def test_related_cli(oi, G, tmp_path):
    from openintel_b200 import store, timeline
    db = str(tmp_path / "fixture.db")
    conn, _, hours = fixture_store(G, db)
    conn.close()
    since, until = T0, T0 + 3600 * len(hours)
    iso = [timeline.format_time(t) for t in (since, until)]
    conn = store.open_store(db)
    with store.MentionIndex(conn) as mi:
        want = json.loads(json.dumps(mi.related(["$AAPL", "calls"], since, until, 5)))
        want_src = json.loads(json.dumps(mi.related(["aapl"], since, until, 20, min_co_mentions=2, source="reddit",
                                                    universe=["calls", "puts", "zzzz"])))
    conn.close()
    assert want[0]["ticker"] == "aapl" and want[0]["mentions"] == 10 and want[0]["related"]
    r = _cli("--store", db, "--since", iso[0], "--until", iso[1], "--top", "5", "$AAPL", "calls")
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout) == {"since": iso[0], "until": iso[1], "source": None, "top": 5, "min_co_mentions": 1,
                                    "universe": None, "anchors": want}
    uni = tmp_path / "universe.txt"
    uni.write_text("calls puts  # options\nzzzz\n", encoding="utf-8")
    r = _cli("--store", db, "--since", iso[0], "--until", iso[1], "--source", "reddit", "--min-co-mentions", "2",
             "--universe", str(uni), "aapl")
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout)
    assert out["anchors"] == want_src and out["min_co_mentions"] == 2 and out["top"] == 20
    # a created_at without an offset: error and exit 1
    bad = make_store(str(tmp_path / "bad.db"), ["gme moon"], ["reddit"], [T0])
    bad.execute("UPDATE posts SET created_at = '2024-01-01 00:00:00'")
    bad.commit()
    bad.close()
    r = _cli("--store", str(tmp_path / "bad.db"), "--since", iso[0], "--until", iso[1], "gme")
    assert r.returncode == 1 and r.stderr.startswith("error:") and "doc_id 0" in r.stderr
    r = _cli("--store", db, "--since", iso[1], "--until", iso[1], "gme")
    assert r.returncode == 2
