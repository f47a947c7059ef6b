"""oi_index_load_post_times / oi_index_mention_timeline and the layers on top (SPEC §8b): the social summary of each
(term, time bucket) must equal the reference's summary over the posts `analyze --mention --since --until` selects, bit
for bit -- unsharded, relayed over the shards of a document-sharded index, and through store.MentionIndex.timeline and
the `timeline` CLI."""
import json
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from mention_util import G, oi  # noqa: F401  (fixtures)
from mention_util import (DAY, ROOT, SMALL_EDGES, T0, fixture_store, iso as _iso, lists, make_store, run_ranks,
                          same_summary, shard_pair, sharded_corpus, small_corpus, synthetic as _synthetic)

pytestmark = pytest.mark.gpu


# ---- 1. the reference fixture: MentionIndex.timeline == analyze_posts over select_posts(mention, since, until) ------
def test_fixture_timeline_equals_analyze_per_bucket(oi, G, tmp_path):
    from openintel_b200 import analyze, capi, store
    conn, mk, hours = fixture_store(G, str(tmp_path / "fixture.db"))
    n = len(hours)
    layouts = [[T0, T0 + 3600 * n],  # one bucket around all posts
               [T0 + 3600 * h for h in range(n + 1)],  # one post per bucket, every post on an edge
               [T0 - 7200, T0 + 1800, T0 + 3600 * 3, T0 + 3600 * 3 + 1, T0 + 3600 * 6 + 59],  # cuts at both ends, an empty bucket
               [T0 + 3600 * 20, T0 + 3600 * 30]]  # no post at all
    with store.MentionIndex(conn) as mi, capi.GpuLexicon() as lx:
        for edges in layouts:
            for src in (None, "reddit", "bluesky"):
                got = mi.timeline(["$AAPL", "calls", "zzzz"], edges, source=src)
                assert len(got) == 3 and all(len(g) == len(edges) - 1 for g in got)
                for word, blocks in zip(("$aapl", "calls", "zzzz"), got):
                    for b, block in enumerate(blocks):
                        _, s, t = analyze.select_posts(conn, source=src, mention=word, since=edges[b], until=edges[b + 1])
                        want = analyze.analyze_posts(lx, s, t, mk)[0]["social"]
                        assert json.dumps(block) == json.dumps(want), (edges, src, word, b)
        assert sum(b["total_mentions"] for b in mi.timeline(["aapl"], layouts[1])[0]) == 10
    conn.close()


# ---- 2. one bucket around all posts == oi_index_mention_summary, bit for bit ---------------------------------------
def test_one_bucket_equals_mention_summary(oi):
    from openintel_b200 import capi
    texts, sources, _ = _synthetic(30_000, 17, n_tickers=80)
    times = T0 + np.random.default_rng(3).integers(0, 30 * DAY, len(texts))
    with capi.GpuLexicon() as lx:
        pol, spec, _, _ = lx.analyze(texts)
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        vocab = ix.build_bm25_text(texts)
        ix.load_post_signals(pol, spec, [0 if s == "reddit" else 1 for s in sources])
        ix.load_post_times(times)
        ids = np.arange(len(vocab), dtype=np.uint32)
        for src in (None, 0, 1):
            s_sum, m_sum = ix.mention_summary(ids, source=src)
            s_tl, m_tl = ix.mention_timeline(ids, [T0, T0 + 30 * DAY], source=src)
            assert s_tl.shape == (len(ids), 1) and s_tl[:, 0].tobytes() == s_sum.tobytes()
            for a, b in zip(m_tl, m_sum):
                same_summary(a[0], b)


# ---- 3. a synthetic corpus with times not in doc order, against the oracle -----------------------------------------
N_SYN = 200_000


@pytest.fixture(scope="module")
def synthetic(oi, tmp_path_factory):
    from openintel_b200 import hostlib, store
    texts, sources, tickers = _synthetic(N_SYN, 2024)
    rng = np.random.default_rng(77)
    times = T0 + rng.integers(-2 * DAY, 367 * DAY, N_SYN)
    on_edge = rng.random(N_SYN) < 0.1
    times[on_edge] = T0 + DAY * rng.integers(-1, 367, int(on_edge.sum()))  # posts exactly on the daily edges
    times[(times >= T0 + 100 * DAY) & (times < T0 + 103 * DAY)] -= 5 * DAY  # three empty days
    conn = make_store(str(tmp_path_factory.mktemp("timeline") / "syn.db"), texts, sources, times)
    scores = [O.lexicon_score(t) for t in texts]
    posts_of = {}
    for d, t in enumerate(texts):
        for w in set(hostlib.tokenize(t)):
            posts_of.setdefault(w, []).append(d)
    mi = store.MentionIndex(conn)
    mi.timeline(["x"], [0, 1])  # loads the post times
    yield dict(conn=conn, mi=mi, tickers=tickers, times=times,
               pol=np.array([s[0] for s in scores], dtype=np.float64), spec=np.array([s[1] for s in scores], dtype=np.int32),
               src=np.array([0 if s == "reddit" else 1 for s in sources], dtype=np.int64),
               posts_of={w: np.array(v, dtype=np.int64) for w, v in posts_of.items()})
    mi.close()
    conn.close()


LAYOUTS = {1: [T0 + 5 * DAY + 1, T0 + 300 * DAY],
           24: [T0 + 15 * DAY * k for k in range(25)],
           365: [T0 + DAY * k for k in range(366)]}


def _check(S, ids, words, sums, states, edges, src, thr):
    for i, w in enumerate(words):
        d = S["posts_of"][w]
        if src is not None:
            d = d[S["src"][d] == src]
        b = np.searchsorted(edges, S["times"][d], side="right") - 1
        for k in range(len(edges) - 1):
            dk = d[b == k]  # doc order kept
            same_summary(sums[i][k], O.social_summary(S["pol"][dk], S["spec"][dk], thr), (w, k, src, thr))
            assert int(states[i, k]["total"]) == len(dk)
            assert [int(states[i, k]["by_source"][s]) for s in (0, 1)] == [int(np.sum(S["src"][dk] == s)) for s in (0, 1)]


@pytest.mark.parametrize("n_buckets", [1, 24, 365])
def test_timeline_equals_the_oracle_over_the_selected_posts(oi, synthetic, n_buckets):
    S = synthetic
    mi = S["mi"]
    edges = LAYOUTS[n_buckets]
    t = S["times"]
    assert (t < edges[0]).any() and (t >= edges[-1]).any() and np.isin(t, edges).sum() > 20
    words = [w for w in S["tickers"] if w in mi.term_id] + ["calls", "puts", "ko", "di"]
    ids = [mi.term_id[w] for w in words]
    ids += ids[:5] + [ids[0]] * 2  # duplicated ids: each gets its own outputs
    words += words[:5] + [words[0]] * 2
    for src in (None, 0, 1):
        for thr in (0.2, 0.99):
            states, sums = mi.ix.mention_timeline(ids, edges, source=src, threshold=thr)
            _check(S, ids, words, sums, states, edges, src, thr)
    if n_buckets == 365:
        head = S["tickers"][0]
        sums = mi.ix.mention_timeline([mi.term_id[head]], edges)[1][0]
        assert [sums[k]["total"] for k in (100, 101, 102)] == [0, 0, 0] and sums[99]["total"] > 0
    # a larger call grows the handle's buffers; the results do not change
    states, _ = mi.ix.mention_timeline(ids, edges, source=1)
    assert mi.ix.mention_timeline(ids * 3, edges, source=1)[0].tobytes() == np.concatenate([states] * 3).tobytes()


# ---- 4. the sharded relay over gloo ranks (all on device 0) -------------------------------------------------------
EDGES_SHARD = [T0 + 6 * 3600 * k for k in range(29)]  # 7 days in 6-hour buckets, posts over 8 days


def _relay_worker(dist, path, tickers):
    from openintel_b200 import store
    conn = store.open_store(path)
    with store.MentionIndex(conn, dist) as mi:
        try:
            out = {src: json.dumps(mi.timeline(tickers, EDGES_SHARD, source=src)) for src in (None, "reddit", "bluesky")}
        except ValueError as e:
            out = "ValueError: %s" % e
    conn.close()
    return out


@pytest.mark.parametrize("world,tokenless", [(2, False), (3, False), (3, True)])
def test_relay_over_the_shards_equals_the_unsharded_timeline(oi, tmp_path, world, tokenless):
    from openintel_b200 import store
    texts, sources, tickers = sharded_corpus(7 + world, world, tokenless)
    times = T0 + np.random.default_rng(world).integers(-DAY, 8 * DAY, len(texts))
    path = str(tmp_path / "posts.db")
    make_store(path, texts, sources, times).close()
    ask = ["$" + t.upper() for t in tickers[:40]] + ["onlyfirst", "calls", "$nothere", tickers[0]]
    conn = store.open_store(path)
    with store.MentionIndex(conn) as mi:
        want = {src: json.dumps(mi.timeline(ask, EDGES_SHARD, source=src)) for src in (None, "reddit", "bluesky")}
    conn.close()
    for rank, got in run_ranks(world, _relay_worker, path, ask):
        assert got == want, rank


def test_a_bad_time_on_one_shard_raises_on_every_rank(oi, tmp_path):
    """a created_at without an offset on the last shard: every rank raises instead of waiting in the relay, and
    reports() does not read the times at all"""
    from openintel_b200 import store
    texts, sources, tickers = _synthetic(600, 5, n_tickers=20)
    path = str(tmp_path / "posts.db")
    conn = make_store(path, texts, sources, T0 + np.arange(600) * 60)
    conn.execute("UPDATE posts SET created_at = '2024-01-01T00:00:00' WHERE doc_id = 555")
    conn.commit()
    with store.MentionIndex(conn) as mi:
        assert mi.reports([tickers[0]])[0]["social"]["total_mentions"] > 0
        with pytest.raises(ValueError) as e:
            mi.timeline([tickers[0]], [T0, T0 + DAY])
        assert "doc_id 555" in str(e.value)
    conn.close()
    res = run_ranks(2, _relay_worker, path, [tickers[0]])
    assert res[1][1].startswith("ValueError") and "doc_id 555" in res[1][1]
    assert res[0][1].startswith("ValueError") and "another shard" in res[0][1]


# ---- 5. the carry by hand: two GpuIndex shards ---------------------------------------------------------------------
def test_carry_continues_the_chain_across_two_shards(oi):
    texts, sources, tickers = _synthetic(20_000, 99, n_tickers=50)
    cut = 12_345
    full, (a, b), vocab, pol, spec = shard_pair(oi, texts, sources, cut)
    times = T0 + np.random.default_rng(1).integers(0, 10 * DAY, len(texts))
    full.load_post_times(times)
    a.load_post_times(times[:cut])
    b.load_post_times(times[cut:])
    edges = [T0 + DAY, T0 + 2 * DAY, T0 + 2 * DAY + 1, T0 + 5 * DAY, T0 + 9 * DAY]
    ids = [vocab.index(t) for t in tickers[:30] if t in vocab] + [vocab.index("calls")]
    srcs = np.array([0 if s == "reddit" else 1 for s in sources])
    to, di = lists(full)
    for src in (None, 0, 1):
        s_all, m_all = full.mention_timeline(ids, edges, source=src)
        s_a, m_a = a.mention_timeline(ids, edges, source=src)
        s_b, m_b = b.mention_timeline(ids, edges, source=src, carry=s_a)
        assert s_b.tobytes() == s_all.tobytes()
        for x, y in zip(m_b, m_all):
            for xk, yk in zip(x, y):
                same_summary(xk, yk)
        # the first shard's summary is the summary of the prefix
        for i, t in enumerate(ids):
            d = di[to[t]:to[t + 1]]
            d = d[d < cut]
            if src is not None:
                d = d[srcs[d] == src]
            bk = np.searchsorted(edges, times[d], side="right") - 1
            for k in range(len(edges) - 1):
                dk = d[bk == k]
                same_summary(m_a[i][k], O.social_summary(pol[dk], spec[dk].astype(np.int32)), (t, k, src))
    for ix in (full, a, b):
        ix.close()


# ---- 6. errors and state --------------------------------------------------------------------------------------------
def _raw_call(ix, terms, n, edges, nb, source=-1, carry=None, out_state=None, out_sum=None):
    from openintel_b200 import capi
    return ix.L.oi_index_mention_timeline(ix.h, capi._addr(terms), n, capi._addr(edges), nb, source, 0.2, capi._addr(carry),
                                          capi._addr(out_state), capi._addr(out_sum))


def test_errors_and_state(oi):
    from openintel_b200 import capi
    texts, pol, spec, src, times = small_corpus()
    edges = SMALL_EDGES
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        vocab = ix.build_bm25_text(texts)
        ix.load_post_signals(pol, spec, src)
        with pytest.raises(ValueError):
            ix.load_post_times(times[:-1])
        assert ix.L.oi_index_load_post_times(ix.h, None) == 1
        ix.load_post_times(times)
        gme, amc = vocab.index("gme"), vocab.index("amc")
        s0, m0 = ix.mention_timeline([gme, amc, gme], edges)
        # gme: posts 0 (hour 50: after the last edge), 1 (hour 10), 4 (hour 40); amc: posts 2 (hour 20), 5 (hour 0)
        assert [[m["total"] for m in row] for row in m0] == [[1, 1], [2, 0], [1, 1]]
        assert s0[0].tobytes() == s0[2].tobytes()
        assert [[m["total"] for m in row] for row in ix.mention_timeline([gme], [T0, T0 + 3 * DAY])[1]] == [[3]]
        assert ix.mention_timeline([], edges)[1] == []
        # refusals; each one writes nothing and the next call gives the same results
        terms = np.array([gme, amc], dtype=np.uint32)
        e64 = np.array(edges, dtype=np.int64)
        big_n = 65537  # x 65536 buckets > 2^32 - 1 keys
        bad = [dict(terms=None), dict(edges=None), dict(out_sum=None), dict(nb=0),
               dict(edges=np.array([T0, T0, T0 + 1], dtype=np.int64)), dict(edges=np.array([T0, T0 + 5, T0 + 4], dtype=np.int64)),
               dict(terms=np.array([gme, len(vocab)], dtype=np.uint32)), dict(terms=np.array([gme, 2 ** 32 - 1], dtype=np.uint32)),
               dict(source=2), dict(source=-2),
               dict(terms=np.zeros(big_n, dtype=np.uint32), n=big_n, edges=T0 + np.arange(65537, dtype=np.int64), nb=65536)]
        for kw in bad:
            out_s = np.full((2, 2), 7, dtype=capi.SOCIAL_SUMMARY_DTYPE)
            out_st = np.full((2, 2), 7, dtype=capi.MENTION_STATE_DTYPE)
            args = dict(terms=terms, n=2, edges=e64, nb=2, out_state=out_st, out_sum=out_s)
            args.update(kw)
            assert _raw_call(ix, **args) == 1, kw
            if args["n"] == big_n:
                assert "2^32 - 1" in capi.load_library().oi_last_error(ix.h).decode()
            if args["out_sum"] is not None:
                assert (out_s.view(np.uint8) == np.full((2, 2), 7, dtype=capi.SOCIAL_SUMMARY_DTYPE).view(np.uint8)).all(), kw
            assert ix.mention_timeline([gme, amc, gme], edges)[0].tobytes() == s0.tobytes(), kw
        # n_terms == 0 is a no-op, even with NULL pointers
        assert _raw_call(ix, None, 0, None, 0) == 0
        # finalize, a rebuilt BM25 part and reloaded signals keep the times
        ix.bm25_finalize()
        assert ix.mention_timeline([gme, amc, gme], edges)[0].tobytes() == s0.tobytes()
        assert ix.build_bm25_text(texts) == vocab
        assert ix.mention_timeline([gme, amc, gme], edges)[0].tobytes() == s0.tobytes()
        ix.load_post_signals(pol, spec, src)
        assert ix.mention_timeline([gme, amc, gme], edges)[0].tobytes() == s0.tobytes()
        # new times move the posts
        ix.load_post_times(times + 24 * 3600)
        assert [[m["total"] for m in row] for row in ix.mention_timeline([gme], edges)[1]] == [[0, 1]]


# ---- 7. the timeline CLI equals `analyze --mention --since --until` per bucket --------------------------------------
def _cli(module, *args):
    out = subprocess.run([sys.executable, "-m", "openintel_b200." + module] + list(args), cwd=ROOT, capture_output=True,
                         text=True, timeout=300)
    return out


def test_timeline_cli_equals_analyze_per_bucket(oi, G, tmp_path):
    db = str(tmp_path / "fixture.db")
    conn, _, hours = fixture_store(G, db)
    conn.close()
    m = G["fixture_posts"]["mock_market"]
    snap = "%r,%r,%d,%d,%r" % (m["last_price"], m["previous_close"], m["volume"], m["avg_volume"], m["iv_rank"])
    since, until = _iso(T0 - 3600), _iso(T0 + 3600 * 9 + 1800)
    r = _cli("timeline", "--store", db, "--since", since, "--until", until, "--every", "4h", "$AAPL", "calls", "zzzz")
    assert r.returncode == 0, r.stderr[-2000:]
    out = json.loads(r.stdout)
    assert set(out) == {"source", "every", "buckets", "tickers"} and out["source"] is None and out["every"] == "4h"
    assert out["buckets"] == [[_iso(T0 - 3600), _iso(T0 + 3 * 3600)], [_iso(T0 + 3 * 3600), _iso(T0 + 7 * 3600)],
                              [_iso(T0 + 7 * 3600), until]]
    assert [t["ticker"] for t in out["tickers"]] == ["$AAPL", "calls", "zzzz"]
    for a, b in out["buckets"]:
        want = _cli("analyze", "--store", db, "--mention", "$AAPL", "--since", a, "--until", b, "--market", snap)
        assert want.returncode == 0, want.stderr[-2000:]
        k = out["buckets"].index([a, b])
        assert json.dumps(out["tickers"][0]["timeline"][k]) == json.dumps(json.loads(want.stdout)["social"])
    assert sum(b["total_mentions"] for b in out["tickers"][0]["timeline"]) == 10
    assert all(b["total_mentions"] == 0 for b in out["tickers"][2]["timeline"])
    r = _cli("timeline", "--store", db, "--since", since, "--until", until, "--every", "1d", "--source", "reddit", "aapl")
    assert r.returncode == 0 and json.loads(r.stdout)["tickers"][0]["timeline"][0]["mentions_by_source"] == {"reddit": 4}
    # errors: stderr and exit 1 for a bad store row, usage errors for bad arguments
    conn = make_store(str(tmp_path / "bad.db"), ["gme moon"], ["reddit"], [T0])
    conn.execute("UPDATE posts SET created_at = '2024-01-01 00:00:00'")
    conn.commit()
    conn.close()
    r = _cli("timeline", "--store", str(tmp_path / "bad.db"), "--since", since, "--until", until, "--every", "1h", "gme")
    assert r.returncode == 1 and "doc_id 0" in r.stderr
    r = _cli("timeline", "--store", db, "--since", until, "--until", since, "--every", "1h", "gme")
    assert r.returncode == 2
