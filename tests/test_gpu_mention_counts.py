"""oi_index_mention_counts and the layers on top (SPEC §8c): the count of every (term, time bucket) must equal the
`total` of oi_index_mention_timeline and a host count over the tokenized posts -- unsharded and summed over the shards of
a document-sharded index -- and store.MentionIndex.trending and the `trending` CLI must rank the terms by the §8c rule,
with the social blocks of `analyze --mention --since --until` for the baseline and the window."""
import json
import math
import subprocess
import sys

import numpy as np
import pytest

from mention_util import G, oi  # noqa: F401  (fixtures)
from mention_util import (DAY, ROOT, SMALL_EDGES, T0, bits as _bits, fixture_store, make_store, run_ranks, sharded_corpus,
                          small_corpus, synthetic as _synthetic)

pytestmark = pytest.mark.gpu

SOURCES = (None, "reddit", "bluesky")


class HostCounts:
    """the host oracle: per post, the set of its tokens (hostlib.tokenize) and its created_at (store.parse_created_at),
    read back from the store; count(t, b) = the posts whose set holds t and whose time is in bucket b"""

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

    def counts(self, edges, source=None):
        nb = len(edges) - 1
        t = self.times[self.docs]
        b = np.searchsorted(np.asarray(edges, dtype=np.int64), t, side="right") - 1
        keep = (b >= 0) & (b < nb)
        if source is not None:
            keep &= self.src[self.docs] == source
        out = np.zeros((self.n_terms, nb), dtype=np.int64)
        np.add.at(out, (self.terms[keep], b[keep]), 1)
        return out


def _timeline_totals(ix, edges, source):
    """the `total` of oi_index_mention_timeline's state for every (term, bucket), all terms in one call"""
    from openintel_b200 import capi
    ids = np.arange(ix.n_terms, dtype=np.uint32)
    e = np.ascontiguousarray(edges, dtype=np.int64)
    nb = len(e) - 1
    states = np.zeros(len(ids) * nb, dtype=capi.MENTION_STATE_DTYPE)
    sums = np.zeros(len(ids) * nb, dtype=capi.SOCIAL_SUMMARY_DTYPE)
    ix._ck(ix.L.oi_index_mention_timeline(ix.h, capi._addr(ids), len(ids), capi._addr(e), nb,
                                          -1 if source is None else int(source), 0.2, None, capi._addr(states),
                                          capi._addr(sums)))
    return states["total"].reshape(len(ids), nb).astype(np.int64)


def _check_counts(mi, oracle, edges):
    from openintel_b200 import store
    for src in SOURCES:
        code = None if src is None else store.SOURCES.index(src)
        got = mi.mention_counts(edges, src)  # loads the post times on the first call
        raw = mi.ix.mention_counts(edges, code)
        assert raw.dtype == np.uint32 and raw.shape == (len(mi.vocab), len(edges) - 1)
        assert got.dtype == np.int64 and (got == raw).all()
        assert (got == _timeline_totals(mi.ix, edges, code)).all(), (edges[:3], src)
        assert (got == oracle.counts(edges, src)).all(), (edges[:3], src)


# ---- 1 + 2. counts == the timeline totals == the host oracle -------------------------------------------------------
def test_fixture_counts_equal_timeline_totals_and_the_host_oracle(oi, G, tmp_path):
    from openintel_b200 import store
    conn, _, hours = fixture_store(G, str(tmp_path / "fixture.db"))
    n = len(hours)
    layouts = [[T0, T0 + 3600 * n],  # one bucket around all posts
               [T0 + 3600 * h for h in range(n + 1)],  # one post per bucket, every post on an edge
               [T0 - 7200, T0 + 1800, T0 + 3600 * 3, T0 + 3600 * 3 + 1, T0 + 3600 * 6 + 59],  # cuts at both ends, an empty bucket
               [T0 + 3600 * 20, T0 + 3600 * 30]]  # no post at all
    with store.MentionIndex(conn) as mi:
        oracle = HostCounts(conn, mi.vocab)
        for edges in layouts:
            _check_counts(mi, oracle, edges)
        aapl = mi.term_id["aapl"]
        assert int(mi.mention_counts(layouts[0])[aapl, 0]) == 10
        assert not mi.mention_counts(layouts[3]).any()
    conn.close()


N_SYN = 200_000


@pytest.fixture(scope="module")
def synthetic(oi, tmp_path_factory):
    from openintel_b200 import store
    texts, sources, tickers = _synthetic(N_SYN, 2025)
    rng = np.random.default_rng(78)
    times = T0 + rng.integers(-2 * DAY, 367 * DAY, N_SYN)
    on_edge = rng.random(N_SYN) < 0.1
    times[on_edge] = T0 + DAY * rng.integers(-1, 367, int(on_edge.sum()))  # posts exactly on the daily edges
    times[(times >= T0 + 100 * DAY) & (times < T0 + 103 * DAY)] -= 5 * DAY  # three empty days
    conn = make_store(str(tmp_path_factory.mktemp("counts") / "syn.db"), texts, sources, times)
    mi = store.MentionIndex(conn)
    yield dict(conn=conn, mi=mi, oracle=HostCounts(conn, mi.vocab), tickers=tickers)
    mi.close()
    conn.close()


SYN_LAYOUTS = {"one": [T0 - 3 * DAY, T0 + 368 * DAY],
               "daily": [T0 + DAY * k for k in range(366)],  # posts on the edges; days 100-102 are empty
               "empty_bucket": [T0 + 99 * DAY, T0 + 100 * DAY, T0 + 103 * DAY, T0 + 110 * DAY],
               "nothing_inside": [T0 - 30 * DAY, T0 - 20 * DAY],
               "hourly_4200": [T0 + 3600 * k for k in range(4201)]}  # too many edges for shared memory


@pytest.mark.parametrize("layout", sorted(SYN_LAYOUTS))
def test_synthetic_counts_equal_timeline_totals_and_the_host_oracle(oi, synthetic, layout):
    S = synthetic
    edges = SYN_LAYOUTS[layout]
    _check_counts(S["mi"], S["oracle"], edges)
    if layout == "daily":
        head = S["mi"].term_id[S["tickers"][0]]
        c = S["mi"].mention_counts(edges)
        assert c[head, 100:103].tolist() == [0, 0, 0] and c[head, 99] > 0
    if layout == "nothing_inside":
        assert not S["mi"].mention_counts(edges).any()


def test_synthetic_trending_equals_the_rule_over_the_host_counts(oi, synthetic):
    S = synthetic
    mi, oracle = S["mi"], S["oracle"]
    t0, t1, t2 = T0 + 200 * DAY, T0 + 230 * DAY, T0 + 233 * DAY
    for src in (None, "bluesky"):
        got = mi.trending(t1, t2, t0, 25, min_mentions=3, source=src)
        cnt = oracle.counts([t0, t1, t2], src)
        assert [(e["ticker"], e["baseline_mentions"], e["mentions"], _bits(e["expected"]), _bits(e["surge"])) for e in got] == \
            [(mi.vocab[t], m, c, _bits(x), _bits(s)) for t, m, c, x, s in _rule(cnt[:, 1], cnt[:, 0], t0, t1, t2, 25, 3)]


# ---- 3. the sharded index: the shards' counts summed over gloo ranks (all on device 0) ------------------------------
E_SHARD = [T0 - DAY, T0 + 3 * DAY, T0 + 6 * DAY, T0 + 7 * DAY, T0 + 9 * DAY]


def _sharded_worker(dist, path):
    from openintel_b200 import store
    conn = store.open_store(path)
    with store.MentionIndex(conn, dist) as mi:
        out = {"counts": {str(src): mi.mention_counts(E_SHARD, src).tolist() for src in SOURCES},
               "trending": {str(src): json.dumps(mi.trending(T0 + 6 * DAY, T0 + 7 * DAY, T0, 15, source=src))
                            for src in SOURCES},
               "universe": json.dumps(mi.trending(T0 + 6 * DAY, T0 + 7 * DAY, T0, 5, universe=["onlyfirst", "$CALLS", "nope"]))}
    conn.close()
    return out


@pytest.mark.parametrize("world,tokenless", [(2, False), (3, False), (3, True)])
def test_sharded_counts_and_trending_equal_the_unsharded_ones(oi, tmp_path, world, tokenless):
    """the sharded corpus of mention_util.sharded_corpus: `onlyfirst` on the first shard only, a token-free middle
    shard with `tokenless`"""
    from openintel_b200 import store
    texts, sources, _ = sharded_corpus(17 + world, world, tokenless)
    times = T0 + np.random.default_rng(world).integers(-2 * DAY, 10 * DAY, len(texts))
    times[[3, 10]] = T0 + 6 * DAY + 5  # onlyfirst: two posts in the window, none in the baseline
    path = str(tmp_path / "posts.db")
    make_store(path, texts, sources, times).close()
    conn = store.open_store(path)
    with store.MentionIndex(conn) as mi:
        want = {"counts": {str(src): mi.mention_counts(E_SHARD, src).tolist() for src in SOURCES},
                "trending": {str(src): json.dumps(mi.trending(T0 + 6 * DAY, T0 + 7 * DAY, T0, 15, source=src)) for src in SOURCES},
                "universe": json.dumps(mi.trending(T0 + 6 * DAY, T0 + 7 * DAY, T0, 5, universe=["onlyfirst", "$CALLS", "nope"]))}
        ranked = {e["ticker"]: e for e in json.loads(want["universe"])}
        assert set(ranked) == {"onlyfirst", "calls"} and ranked["onlyfirst"]["surge"] == 2.0  # m = 0: surge = c
    conn.close()
    for rank, got in run_ranks(world, _sharded_worker, path):
        assert got == want, rank


# ---- 4. trending over planted surges ----------------------------------------------------------------------------------
TB, TW, TE = T0, T0 + 7 * DAY, T0 + 8 * DAY  # baseline [TB, TW), window [TW, TE)


def _rule(c, m, t0, t1, t2, k, min_mentions, allowed=None):
    """SPEC §8c in plain Python floats: [(term id, m, c, expected, surge)] in rank order"""
    rows = []
    for t in range(len(c)):
        if c[t] >= min_mentions and (allowed is None or t in allowed):
            e = (float(int(m[t])) * float(t2 - t1)) / float(t1 - t0)
            rows.append((t, int(m[t]), int(c[t]), e, (float(int(c[t])) - e) / math.sqrt(e + 1.0)))
    rows.sort(key=lambda r: (-r[4], r[0]))
    return rows[:k]


@pytest.fixture(scope="module")
def planted(oi, G, tmp_path_factory):
    from openintel_b200 import fusion, hostlib, store
    n = 6000
    texts, sources, tickers = _synthetic(n, 31, n_tickers=80)
    rng = np.random.default_rng(32)
    times = TB - DAY + rng.integers(0, 10 * DAY, n)  # posts from a day before the baseline to two days after the window
    mentions = [set(hostlib.tokenize(t)) for t in texts]
    surging = [tickers[5], tickers[9], tickers[20]]
    for j, w in enumerate(surging):  # most of their posts move into the window
        d = [i for i in range(n) if w in mentions[i]]
        move = np.random.default_rng(40 + j).random(len(d)) < (0.8, 0.6, 0.5)[j]
        for i, mv in zip(d, move):
            if mv:
                times[i] = TW + (i * 7919) % DAY
    # two tickers with identical (c, m) = (6, 3), and one that appears in the window only
    for word, posts in (("twina", range(100, 109)), ("twinb", range(200, 209)), ("newbie", range(300, 305))):
        for j, i in enumerate(posts):
            texts[i] += " " + word
            times[i] = (TB + DAY * j + 11 if (word != "newbie" and j < 3) else TW + 3600 * j + 7)
    path = str(tmp_path_factory.mktemp("planted") / "planted.db")
    conn = make_store(path, texts, sources, times)
    mi = store.MentionIndex(conn)
    m = G["fixture_posts"]["mock_market"]
    mk = fusion.MarketSummary.from_snapshot(m["last_price"], m["previous_close"], m["volume"], m["avg_volume"], m["iv_rank"])
    yield dict(conn=conn, path=path, mi=mi, oracle=HostCounts(conn, mi.vocab), surging=surging, mk=mk)
    mi.close()
    conn.close()


def _social(lx, conn, mk, src, word, since, until):
    from openintel_b200 import analyze
    _, s, t = analyze.select_posts(conn, source=src, mention=word, since=since, until=until)
    return analyze.analyze_posts(lx, s, t, mk)[0]["social"]


@pytest.mark.parametrize("src", SOURCES)
def test_trending_over_planted_surges(oi, planted, src):
    from openintel_b200 import capi
    P = planted
    mi, conn = P["mi"], P["conn"]
    cnt = P["oracle"].counts([TB, TW, TE], src)
    for k, mm in ((12, 1), (40, 2), (len(mi.vocab) + 5, 1)):
        got = mi.trending(TW, TE, TB, k, min_mentions=mm, source=src)
        want = _rule(cnt[:, 1], cnt[:, 0], TB, TW, TE, k, mm)
        assert [(mi.term_id[e["ticker"]], e["baseline_mentions"], e["mentions"], _bits(e["expected"]), _bits(e["surge"]))
                for e in got] == [(t, m, c, _bits(x), _bits(s)) for t, m, c, x, s in want], (k, mm)
        assert len(got) == min(k, int(np.count_nonzero(cnt[:, 1] >= mm)))
    got = mi.trending(TW, TE, TB, 12, source=src)
    names = [e["ticker"] for e in got]
    if src is None:
        assert set(names[:3]) == set(P["surging"])
        new = got[names.index("newbie")]
        assert (new["mentions"], new["baseline_mentions"], new["expected"], new["surge"]) == (5, 0, 0.0, 5.0)
        a, b = names.index("twina"), names.index("twinb")
        assert b == a + 1 and got[a]["surge"] == got[b]["surge"] and (got[a]["mentions"], got[a]["baseline_mentions"]) == (6, 3)
    with capi.GpuLexicon() as lx:
        for e in got:
            assert e["social"]["baseline"]["total_mentions"] == e["baseline_mentions"]
            assert e["social"]["window"]["total_mentions"] == e["mentions"]
            assert json.dumps(e["social"]["baseline"]) == json.dumps(_social(lx, conn, P["mk"], src, e["ticker"], TB, TW))
            assert json.dumps(e["social"]["window"]) == json.dumps(_social(lx, conn, P["mk"], src, e["ticker"], TW, TE))
    # a universe: normalised like --mention; entries outside the vocabulary are never ranked
    uni = ["$" + P["surging"][1].upper(), "TwinB", "newbie", "$notaword", "the"]
    got = mi.trending(TW, TE, TB, 10, source=src, universe=uni)
    allowed = {mi.term_id[w] for w in (P["surging"][1], "twinb", "newbie", "the")}
    want = _rule(cnt[:, 1], cnt[:, 0], TB, TW, TE, 10, 1, allowed)
    assert [(e["ticker"], _bits(e["surge"])) for e in got] == [(mi.vocab[t], _bits(s)) for t, _, _, _, s in want]
    assert mi.trending(TW, TE, TB, 10, source=src, universe=[]) == []
    assert mi.trending(TW, TE, TB, 10, source=src, min_mentions=10 ** 6) == []


def test_trending_refuses_bad_windows(oi, planted):
    mi = planted["mi"]
    for args in ((TW, TE, TW, 5), (TW, TE, TE, 5), (TE, TW, TB, 5), (TW, TE, TB, 0)):
        with pytest.raises(ValueError):
            mi.trending(*args)
    with pytest.raises(ValueError):
        mi.trending(TW, TE, TB, 5, min_mentions=0)
    for edges in ([TB], [TB, TB], [TW, TB]):
        with pytest.raises(ValueError):
            mi.mention_counts(edges)


# ---- 5. errors and state ----------------------------------------------------------------------------------------------
def _raw_counts(ix, edges, nb, source=-1, out=None):
    from openintel_b200 import capi
    return ix.L.oi_index_mention_counts(ix.h, capi._addr(edges), nb, source, capi._addr(out))


def test_errors_and_state(oi):
    texts, pol, spec, src, times = small_corpus()
    edges = SMALL_EDGES
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        vocab = ix.build_bm25_text(texts)
        ix.load_post_signals(pol, spec, src)
        ix.load_post_times(times)
        c0 = ix.mention_counts(edges)
        gme, amc, the = vocab.index("gme"), vocab.index("amc"), vocab.index("the")
        # gme: posts 0 (hour 50: after the last edge), 1 (hour 10), 4 (hour 40, "GME GME" counts once); amc: posts 2
        # (hour 20), 5 (hour 0); the: post 0
        assert c0.shape == (len(vocab), 2) and c0[gme].tolist() == [1, 1] and c0[amc].tolist() == [2, 0]
        assert c0[the].tolist() == [0, 0]
        assert ix.mention_counts(edges, 0)[gme].tolist() == [0, 0] and ix.mention_counts(edges, 1)[gme].tolist() == [1, 1]
        assert (c0 == _timeline_totals(ix, edges, None)).all()
        # refusals: each one writes nothing and the next call gives the same counts
        e64 = np.array(edges, dtype=np.int64)
        bad = [dict(edges=None), dict(out=None), dict(nb=0), dict(edges=np.array([T0, T0, T0 + 1], dtype=np.int64)),
               dict(edges=np.array([T0, T0 + 5, T0 + 4], dtype=np.int64)), dict(source=2), dict(source=-2)]
        for kw in bad:
            out = np.full((len(vocab), 2), 7, dtype=np.uint32)
            args = dict(edges=e64, nb=2, out=out)
            args.update(kw)
            assert _raw_counts(ix, **args) == 1, kw
            assert (out == 7).all(), kw
            assert (ix.mention_counts(edges) == c0).all(), kw
        # a larger call grows the handle's buffer; one with a timeline call in between changes nothing
        many = T0 - DAY + 3600 * np.arange(24 * 200 + 1, dtype=np.int64)
        big = ix.mention_counts(many)
        assert big.shape == (len(vocab), 24 * 200) and int(big.sum()) == ix.bm25_local_stats()[2]  # every posting once
        assert ix.mention_timeline([gme], edges)[0].shape == (1, 2)
        assert (ix.mention_counts(edges) == c0).all()
        # before and after finalize, a rebuilt BM25 part and reloaded signals: the same counts
        ix.bm25_finalize()
        assert (ix.mention_counts(edges) == c0).all()
        assert ix.build_bm25_text(texts) == vocab
        assert (ix.mention_counts(edges) == c0).all()
        ix.load_post_signals(pol, spec, src)
        assert (ix.mention_counts(edges) == c0).all()
        # new times move the posts
        ix.load_post_times(times + 24 * 3600)
        assert ix.mention_counts(edges)[gme].tolist() == [0, 1]
    # a shard without a posting: all zeros
    with oi.GpuIndex(n_docs=3, dim=4, max_k=1) as ix:
        ix.load_bm25(np.zeros(5, np.uint64), np.zeros(0, np.uint32), np.zeros(0, np.uint32), np.zeros(3, np.uint32))
        ix.load_post_signals(np.zeros(3), np.zeros(3, np.uint8), np.zeros(3, np.uint8))
        ix.load_post_times(np.full(3, T0, dtype=np.int64))
        out = np.full((4, 2), 7, dtype=np.uint32)
        assert _raw_counts(ix, np.array(edges, dtype=np.int64), 2, out=out) == 0 and not out.any()
        ix.bm25_finalize()
        assert not ix.mention_counts(edges, 1).any()


# ---- 6. the trending CLI prints what MentionIndex.trending returns ---------------------------------------------------
def _cli(*args):
    return subprocess.run([sys.executable, "-m", "openintel_b200.trending"] + list(args), cwd=ROOT, capture_output=True,
                          text=True, timeout=300)


def test_trending_cli(oi, planted, tmp_path):
    from openintel_b200 import timeline
    P = planted
    db, mi = P["path"], P["mi"]
    iso = [timeline.format_time(t) for t in (TB, TW, TE)]
    r = _cli("--store", db, "--baseline-since", iso[0], "--since", iso[1], "--until", iso[2], "--top", "7")
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout)
    assert out == {"baseline_since": iso[0], "since": iso[1], "until": iso[2], "source": None, "top": 7, "min_mentions": 1,
                   "universe": None, "ranked": json.loads(json.dumps(mi.trending(TW, TE, TB, 7)))}
    assert [_bits(e["surge"]) for e in out["ranked"]] == [_bits(e["surge"]) for e in mi.trending(TW, TE, TB, 7)]
    uni = tmp_path / "universe.txt"
    uni.write_text("$%s  # surging\nTWINA twinb\n$NOTAWORD\n" % P["surging"][0].upper(), encoding="utf-8")
    r = _cli("--store", db, "--baseline-since", iso[0], "--since", iso[1], "--until", iso[2], "--source", "reddit",
             "--min-mentions", "2", "--universe", str(uni))
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout)
    assert out["source"] == "reddit" and out["min_mentions"] == 2 and out["universe"] == str(uni) and out["top"] == 20
    assert out["ranked"] == json.loads(json.dumps(mi.trending(TW, TE, TB, 20, min_mentions=2, source="reddit",
                                                              universe=["$" + P["surging"][0], "twina", "twinb", "notaword"])))
    assert {e["ticker"] for e in out["ranked"]} <= {P["surging"][0], "twina", "twinb"}
    # a created_at without an offset: error and exit 1
    conn = make_store(str(tmp_path / "bad.db"), ["gme moon"], ["reddit"], [T0])
    conn.execute("UPDATE posts SET created_at = '2024-01-01 00:00:00'")
    conn.commit()
    conn.close()
    r = _cli("--store", str(tmp_path / "bad.db"), "--baseline-since", iso[0], "--since", iso[1], "--until", iso[2])
    assert r.returncode == 1 and r.stderr.startswith("error:") and "doc_id 0" in r.stderr
    r = _cli("--store", db, "--baseline-since", iso[1], "--since", iso[1], "--until", iso[2])
    assert r.returncode == 2
