"""oi_index_load_post_signals / oi_index_mention_summary and the layers on top (SPEC §8a): the social summary of each
term's posting list must equal the reference's summary over the posts `analyze --mention` selects, bit for bit --
unsharded, relayed over the shards of a document-sharded index, and through store.MentionIndex and the `compare` CLI."""
import json
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from mention_util import G, oi  # noqa: F401  (fixtures)
from mention_util import (ROOT, fixture_store, lists, make_store, run_ranks, same_summary, shard_pair, sharded_corpus,
                          SMALL_EDGES, small_corpus, synthetic as _synthetic)

pytestmark = pytest.mark.gpu


# ---- 1. the reference fixture: MentionIndex.reports == analyze_posts over select_posts(mention=...) -----------------
def test_fixture_reports_equal_analyze_with_mention(oi, G, tmp_path):
    from openintel_b200 import analyze, capi, store
    conn, mk, _ = fixture_store(G, str(tmp_path / "fixture.db"))
    with store.MentionIndex(conn) as mi, capi.GpuLexicon() as lx:
        for src in (None, "reddit", "bluesky"):
            for market in (mk, None):
                got = mi.reports(["$AAPL"], source=src, markets=None if market is None else {"AAPL": market})[0]
                want = analyze.analyze_posts(lx, *analyze.select_posts(conn, source=src, mention="$aapl")[1:], market)[0]
                assert got == want and json.dumps(got) == json.dumps(want), (src, market)
        assert mi.reports(["$AAPL"])[0]["social"]["total_mentions"] == 10
        # a word that is not in the vocabulary has no post: NoData without a market, an empty report with one
        assert mi.reports(["$ZZZZ", "aapl"])[0] is None
        assert mi.reports(["zzzz"], markets={"$ZZZZ": mk}) == [analyze.analyze_posts(lx, [], [], mk)[0]]
    conn.close()


# ---- 2. a synthetic corpus, one batched call per (source, threshold) ----------------------------------------------
N_SYN = 200_000


@pytest.fixture(scope="module")
def synthetic(oi, tmp_path_factory):
    from openintel_b200 import hostlib, store
    texts, sources, tickers = _synthetic(N_SYN, 2024)
    path = str(tmp_path_factory.mktemp("mention") / "syn.db")
    conn = make_store(path, texts, sources)
    scores = [O.lexicon_score(t) for t in texts]
    pol = np.array([s[0] for s in scores], dtype=np.float64)
    spec = np.array([s[1] for s in scores], dtype=np.int32)
    src = np.array([0 if s == "reddit" else 1 for s in sources], dtype=np.int64)
    posts_of = {}  # token -> the posts select_posts(mention=token) keeps, in doc order
    for d, t in enumerate(texts):
        for w in set(hostlib.tokenize(t)):
            posts_of.setdefault(w, []).append(d)
    mi = store.MentionIndex(conn)
    yield dict(conn=conn, mi=mi, texts=texts, tickers=tickers, pol=pol, spec=spec, src=src,
               posts_of={w: np.array(v, dtype=np.int64) for w, v in posts_of.items()})
    mi.close()
    conn.close()


def test_batched_summaries_equal_the_oracle_over_the_selected_posts(oi, synthetic):
    from openintel_b200 import analyze
    S = synthetic
    mi, posts_of = S["mi"], S["posts_of"]
    head = S["tickers"][0]
    assert 0.25 * N_SYN < len(posts_of[head]) < 0.35 * N_SYN  # many 2048-entry tiles
    assert "ko" in posts_of and "di" in posts_of
    # the host model of select_posts is select_posts itself, on a few terms and sources
    for w, src in ((head, None), (S["tickers"][5], "bluesky"), ("ko", "reddit")):
        ids, _, _ = analyze.select_posts(S["conn"], source=src, mention="$" + w.upper())
        want = posts_of[w] if src is None else posts_of[w][S["src"][posts_of[w]] == ("reddit", "bluesky").index(src)]
        assert [int(i[1:]) for i in ids] == want.tolist()
    words = [w for w in S["tickers"] if w in mi.term_id] + ["calls", "puts", "ko", "di"]
    assert len(words) > 250
    ids = [mi.term_id[w] for w in words]
    ids += ids[:7] + [ids[0]] * 3  # duplicated ids: each gets its own output
    words += words[:7] + [words[0]] * 3
    for src in (None, 0, 1):
        for thr in (0.2, 0.0, 0.99):
            states, sums = mi.ix.mention_summary(ids, source=src, threshold=thr)
            for i, w in enumerate(words):
                d = posts_of[w] if src is None else posts_of[w][S["src"][posts_of[w]] == src]
                want = O.social_summary(S["pol"][d], S["spec"][d], thr)
                same_summary(sums[i], want, (w, src, thr))
                assert [int(states[i]["by_source"][s]) for s in (0, 1)] == [int(np.sum(S["src"][d] == s)) for s in (0, 1)]
                assert int(states[i]["total"]) == len(d) and int(states[i]["speculative"]) == int(S["spec"][d].sum())
    # a call too large for a pinned staging slot, and the same call forced onto the large-call path, agree
    big = np.array(ids * 40, dtype=np.uint32)
    s_big, m_big = mi.ix.mention_summary(big, source=1, threshold=0.2)
    mi.ix.set_option("no_pinned_staging", 1)
    s_dir, m_dir = mi.ix.mention_summary(ids, source=1, threshold=0.2)
    mi.ix.set_option("no_pinned_staging", 0)
    s_pin, m_pin = mi.ix.mention_summary(ids, source=1, threshold=0.2)
    assert s_big.tobytes() == np.tile(s_pin, 40).tobytes() and s_dir.tobytes() == s_pin.tobytes()
    for a, b in zip(m_dir, m_pin):
        same_summary(a, b)


# ---- 3. the sharded relay over gloo ranks (all on device 0) -------------------------------------------------------
def _relay_worker(dist, path, tickers):
    from openintel_b200 import store
    conn = store.open_store(path)
    with store.MentionIndex(conn, dist) as mi:
        out = {src: json.dumps(mi.reports(tickers, source=src)) for src in (None, "reddit", "bluesky")}
    conn.close()
    return out


@pytest.mark.parametrize("world,tokenless", [(2, False), (3, False), (3, True)])
def test_relay_over_the_shards_equals_the_unsharded_reports(oi, tmp_path, world, tokenless):
    """every rank's reports equal the unsharded MentionIndex's, bit for bit (mention_util.sharded_corpus)"""
    from openintel_b200 import store
    texts, sources, tickers = sharded_corpus(7 + world, world, tokenless)
    path = str(tmp_path / "posts.db")
    make_store(path, texts, sources).close()
    ask = ["$" + t.upper() for t in tickers[:40]] + ["onlyfirst", "calls", "$nothere", tickers[0]]

    conn = store.open_store(path)
    with store.MentionIndex(conn) as mi:
        want = {src: json.dumps(mi.reports(ask, source=src)) for src in (None, "reddit", "bluesky")}
    conn.close()
    assert '"total_mentions": 2' in want[None]
    for rank, got in run_ranks(world, _relay_worker, path, ask):
        assert got == want, rank


# ---- 4. the carry by hand: two GpuIndex shards ---------------------------------------------------------------------
def test_carry_continues_the_chain_across_two_shards(oi):
    texts, sources, tickers = _synthetic(20_000, 99, n_tickers=50)
    cut = 12_345
    full, (a, b), vocab, pol, spec = shard_pair(oi, texts, sources, cut)
    ids = [vocab.index(t) for t in tickers[:30] if t in vocab] + [vocab.index("calls")]
    for src in (None, 0, 1):
        s_all, m_all = full.mention_summary(ids, source=src)
        s_a, m_a = a.mention_summary(ids, source=src)
        s_b, m_b = b.mention_summary(ids, source=src, carry=s_a)
        assert s_b.tobytes() == s_all.tobytes()
        for x, y in zip(m_b, m_all):
            same_summary(x, y)
        # the first shard's summary is the summary of the prefix
        srcs = np.array([0 if s == "reddit" else 1 for s in sources])
        to, di = lists(full)
        for i, t in enumerate(ids):
            d = di[to[t]:to[t + 1]]
            d = d[d < cut]
            if src is not None:
                d = d[srcs[d] == src]
            same_summary(m_a[i], O.social_summary(pol[d], spec[d].astype(np.int32)), (t, src))
    for ix in (full, a, b):
        ix.close()


# ---- 5. errors and state --------------------------------------------------------------------------------------------
CALLS = {"summary": lambda ix: ix.mention_summary([0]),
         "timeline": lambda ix: ix.mention_timeline([0], SMALL_EDGES),
         "counts": lambda ix: ix.mention_counts(SMALL_EDGES)}
LOADED = ("nothing", "signals", "signals+times", "bm25", "bm25+times", "bm25+signals")


# the summary needs no post times: with the BM25 part and the signals nothing is missing
@pytest.mark.parametrize("call,loaded", [(c, l) for c in sorted(CALLS) for l in LOADED if (c, l) != ("summary", "bm25+signals")])
def test_a_call_before_its_data_is_refused(oi, call, loaded):
    """status 5 (OI_ERR_STATE) naming the first missing piece: the BM25 part, then the signals, then the post times
    (timeline and counts only)"""
    texts, pol, spec, src, times = small_corpus()
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        if "bm25" in loaded:
            ix.build_bm25_text(texts)
        if "signals" in loaded:
            ix.load_post_signals(pol, spec, src)
        if "times" in loaded:
            ix.load_post_times(times)
        with pytest.raises(oi.OiError) as e:
            CALLS[call](ix)
    missing = "BM25" if "bm25" not in loaded else "signals" if "signals" not in loaded else "times"
    assert e.value.status == 5 and missing in e.value.message


def test_errors_and_state(oi):
    texts, pol, spec, src, _ = small_corpus()
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        vocab = ix.build_bm25_text(texts)
        ix.load_post_signals(pol, spec, src)
        gme, amc = vocab.index("gme"), vocab.index("amc")
        s0, m0 = ix.mention_summary([gme, amc, gme])
        assert [m["total"] for m in m0] == [3, 2, 3] and s0[0].tobytes() == s0[2].tobytes()
        assert ix.mention_summary([])[1] == []
        for kw in (dict(term_ids=[len(vocab)]), dict(term_ids=[gme, 2 ** 32 - 1]), dict(term_ids=[gme], source=2),
                   dict(term_ids=[gme], source=-2)):
            with pytest.raises(oi.OiError) as e:
                ix.mention_summary(**kw)
            assert e.value.status == 1, kw
        for bad in (dict(pol=np.nan), dict(pol=1.5), dict(pol=-1.0000000000000002), dict(pol=np.inf), dict(spec=2),
                    dict(src=2), dict(src=255)):
            p, s, c = pol.copy(), spec.copy(), src.copy()
            p[3], s[3], c[3] = bad.get("pol", p[3]), bad.get("spec", s[3]), bad.get("src", c[3])
            with pytest.raises(oi.OiError) as e:
                ix.load_post_signals(p, s, c)
            assert e.value.status == 1 and "post 3" in e.value.message, bad
            # the refused call kept the previous signals
            s1, m1 = ix.mention_summary([gme, amc, gme])
            assert s1.tobytes() == s0.tobytes()
        # -0.0 is stored as +0.0: the same summaries
        p = pol.copy()
        p[p == 0.0] = -0.0
        assert np.signbit(p).sum() > np.signbit(pol).sum()
        ix.load_post_signals(p, spec, src)
        assert ix.mention_summary([gme, amc, gme])[0].tobytes() == s0.tobytes()
        # finalize and a rebuilt BM25 part keep the signals
        ix.bm25_finalize()
        assert ix.mention_summary([gme, amc, gme])[0].tobytes() == s0.tobytes()
        assert ix.build_bm25_text(texts) == vocab
        assert ix.mention_summary([gme, amc, gme])[0].tobytes() == s0.tobytes()
        with pytest.raises(ValueError):
            ix.load_post_signals(pol[:-1], spec[:-1], src[:-1])


# ---- 6. the compare CLI on the fixture store -----------------------------------------------------------------------
def _compare(db, *args):
    out = subprocess.run([sys.executable, "-m", "openintel_b200.compare", "--store", db] + list(args), cwd=ROOT,
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout)


def test_compare_cli_ranks_reports(oi, G, tmp_path):
    from openintel_b200 import store
    db = str(tmp_path / "fixture.db")
    conn, mk, _ = fixture_store(G, db)
    with store.MentionIndex(conn) as mi:
        want = mi.reports(["AAPL", "calls", "zzzz"], markets={"AAPL": mk})
    conn.close()
    m = G["fixture_posts"]["mock_market"]
    snap = "AAPL=%r,%r,%d,%d,%r" % (m["last_price"], m["previous_close"], m["volume"], m["avg_volume"], m["iv_rank"])
    out = _compare(db, "--by", "total_mentions", "--market", snap, "calls", "$AAPL", "zzzz")
    assert set(out) == {"by", "source", "ranked", "no_data"} and out["by"] == "total_mentions" and out["source"] is None
    assert [e["ticker"] for e in out["ranked"]] == ["$AAPL", "calls"] and out["no_data"] == ["zzzz"]
    assert [e["value"] for e in out["ranked"]] == [10, 2]
    assert json.dumps(out["ranked"][0]["report"]) == json.dumps(want[0])
    assert json.dumps(out["ranked"][1]["report"]) == json.dumps(want[1]) and want[2] is None
    # descending by another metric; a tie keeps the order the tickers were given
    out = _compare(db, "--by", "speculation_index", "calls", "aapl", "$AAPL")
    vals = [e["value"] for e in out["ranked"]]
    assert vals == sorted(vals, reverse=True) and vals[0] > vals[1] == vals[2]
    assert [e["ticker"] for e in out["ranked"]] == ["calls", "aapl", "$AAPL"]
    out = _compare(db, "--by", "speculation_index", "$AAPL", "aapl", "calls")
    assert [e["ticker"] for e in out["ranked"]] == ["calls", "$AAPL", "aapl"]
    out = _compare(db, "--source", "reddit", "--by", "net_sentiment", "aapl", "zzzz")
    assert out["source"] == "reddit" and out["ranked"][0]["report"]["social"]["mentions_by_source"] == {"reddit": 4}
    assert out["no_data"] == ["zzzz"]
