"""oi_index_load_post_signals / oi_index_mention_summary and the layers on top (SPEC §8a): the social summary of each
term's posting list must equal the reference's summary over the posts `analyze --mention` selects, bit for bit --
unsharded, relayed over the shards of a document-sharded index, and through store.MentionIndex and the `compare` CLI."""
import json
import os
import socket
import struct
import subprocess
import sys

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("total", "bullish", "bearish", "neutral", "net_sentiment", "speculation_index", "bull_bear_ratio")
BULL = ["moon", "calls", "long", "buy", "bullish", "squeeze", "breakout", "rocket", "pump", "rip", "green", "up", "rally", "bull"]
BEAR = ["puts", "short", "sell", "bearish", "dump", "crash", "drilling", "bagholder", "rug", "red", "down", "tank", "bear"]
JARGON = ["calls", "puts", "0dte", "yolo", "leaps", "theta", "gamma", "squeeze", "otm", "itm", "strike", "iv", "delta", "vega",
          "contracts"]


@pytest.fixture(scope="module")
def oi():
    import __graft_entry__ as ge  # noqa: F401
    import openintel_b200
    openintel_b200.load_library()
    import runpy
    from openintel_b200 import hostlib
    runpy.run_path(os.path.join(os.path.dirname(hostlib.__file__), "host", "build.py"), run_name="__build__")
    return openintel_b200


@pytest.fixture(scope="module")
def G():
    with open(os.path.join(ROOT, "tests", "golden", "reference_lexicon_goldens.json"), encoding="utf-8") as f:
        return json.load(f)


def _bits(x):
    return struct.pack("<d", x)


def _same_summary(a, b, what=""):
    for f in FIELDS:
        if isinstance(b[f], float):
            assert _bits(a[f]) == _bits(b[f]), (what, f, a[f], b[f])
        else:
            assert a[f] == b[f], (what, f, a[f], b[f])


def _posts(texts, sources):
    return [dict(id="p%d" % i, source=s, author="a%d" % (i % 97), text=t, created_at="2024-01-01T00:00:00Z", engagement=i % 50)
            for i, (t, s) in enumerate(zip(texts, sources))]


def _store(path, texts, sources):
    """a store WITHOUT embeddings: the mention path does not need them"""
    from openintel_b200 import store
    conn = store.open_store(path)
    store.insert_posts(conn, _posts(texts, sources))
    return conn


def _fixture(G, path):
    from openintel_b200 import fusion
    fx = G["fixture_posts"]
    conn = _store(path, [p["text"] for p in fx["posts"]], [p["source"] for p in fx["posts"]])
    m = fx["mock_market"]
    return conn, fusion.MarketSummary.from_snapshot(m["last_price"], m["previous_close"], m["volume"], m["avg_volume"], m["iv_rank"])


# ---- 1. the reference fixture: MentionIndex.reports == analyze_posts over select_posts(mention=...) -----------------
def test_fixture_reports_equal_analyze_with_mention(oi, G, tmp_path):
    from openintel_b200 import analyze, capi, store
    conn, mk = _fixture(G, str(tmp_path / "fixture.db"))
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


def _ticker_names(n, rng):
    letters = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz", dtype=np.uint8)
    taken = set(BULL + BEAR + JARGON)
    out = []
    while len(out) < n:
        w = rng.choice(letters, size=int(rng.integers(2, 6))).tobytes().decode()
        if w not in taken:
            taken.add(w)
            out.append(w)
    return out


def _synthetic(n_posts, seed, n_tickers=300):
    """posts of lexicon words, Zipf-distributed tickers ($GME / Gme / gme) and filler; a head ticker in ~30 % of the
    posts; posts without a lexicon hit, posts with as many bull as bear hits, a few KELVIN SIGN / U+0130 posts"""
    rng = np.random.default_rng(seed)
    tickers = _ticker_names(n_tickers, rng)
    filler = ["w%d" % i for i in range(500)] + ["the", "and", "to", "of", "is"]
    lex = BULL + BEAR + JARGON
    p = 1.0 / np.arange(1, n_tickers) ** 1.1  # tickers[0] is the head ticker, the others are Zipf-distributed
    n_lex, n_tick, n_fill = rng.integers(0, 4, n_posts), rng.integers(0, 3, n_posts), rng.integers(1, 8, n_posts)
    lex_w = rng.integers(0, len(lex), int(n_lex.sum()))
    tick_w = 1 + rng.choice(n_tickers - 1, size=int(n_tick.sum()), p=p / p.sum())
    fill_w = rng.integers(0, len(filler), int(n_fill.sum()))
    has_head = rng.random(n_posts) < 0.3
    keys = rng.random(int(n_lex.sum() + n_tick.sum() + n_fill.sum() + has_head.sum()) + 4 * n_posts)
    li = ti = fi = ki = 0
    texts = []
    for i in range(n_posts):
        words = []
        kind = i % 10
        if kind < 7:
            words += [lex[j] for j in lex_w[li:li + n_lex[i]]]
        elif kind == 7:
            words += ["moon", "dump"] if i % 20 == 7 else ["calls", "puts", "buy", "sell"]  # bull == bear
        # kind 8, 9: no lexicon word at all
        li += n_lex[i]
        tw = [tickers[t] for t in tick_w[ti:ti + n_tick[i]]] + ([tickers[0]] if has_head[i] else [])
        ti += n_tick[i]
        words += [("$" + w.upper(), w.capitalize(), w)[(i + j) % 3] for j, w in enumerate(tw)]
        words += [filler[j] for j in fill_w[fi:fi + n_fill[i]]]
        fi += n_fill[i]
        order = np.argsort(keys[ki:ki + len(words)])
        ki += len(words)
        t = " ".join(words[j] for j in order) + ("!" if i % 3 else "")
        if i % 997 == 0:
            t += " \u212aO D\u0130P bul\u0130sh"  # -> "ko", "di", "p", "buli", "sh" (SPEC §6)
        texts.append(t)
    sources = [("reddit", "bluesky")[int(b)] for b in rng.integers(0, 2, size=n_posts)]
    return texts, sources, tickers


@pytest.fixture(scope="module")
def synthetic(oi, tmp_path_factory):
    from openintel_b200 import hostlib, store
    texts, sources, tickers = _synthetic(N_SYN, 2024)
    path = str(tmp_path_factory.mktemp("mention") / "syn.db")
    conn = _store(path, texts, sources)
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
                _same_summary(sums[i], want, (w, src, thr))
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
        _same_summary(a, b)


# ---- 3. the sharded relay over gloo ranks (all on device 0) -------------------------------------------------------
N_SHARD = 3000


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _relay_worker(rank, world, port, path, tickers, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from openintel_b200 import store
        conn = store.open_store(path)
        with store.MentionIndex(conn, dist) as mi:
            out = {src: json.dumps(mi.reports(tickers, source=src)) for src in (None, "reddit", "bluesky")}
        conn.close()
        q.put((rank, out))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,tokenless", [(2, False), (3, False), (3, True)])
def test_relay_over_the_shards_equals_the_unsharded_reports(oi, tmp_path, world, tokenless):
    """every rank's reports equal the unsharded MentionIndex's, bit for bit.  `onlyfirst` appears on the first shard
    only; with `tokenless`, the middle shard's posts hold no token at all (its lists are all empty)."""
    import torch.multiprocessing as mp
    from openintel_b200 import sharding, store
    texts, sources, tickers = _synthetic(N_SHARD, 7 + world, n_tickers=60)
    texts[3] += " onlyfirst moon"
    texts[10] += " onlyfirst dump"
    if tokenless:
        base, n = sharding.shard_range(N_SHARD, world, 1)
        for i in range(base, base + n):
            texts[i] = ("!!!", "ÿþ ???", "... — !!", "\U0001f680 $$")[i % 4]
    path = str(tmp_path / "posts.db")
    _store(path, texts, sources).close()
    ask = ["$" + t.upper() for t in tickers[:40]] + ["onlyfirst", "calls", "$nothere", tickers[0]]

    conn = store.open_store(path)
    with store.MentionIndex(conn) as mi:
        want = {src: json.dumps(mi.reports(ask, source=src)) for src in (None, "reddit", "bluesky")}
    conn.close()
    assert '"total_mentions": 2' in want[None]

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_relay_worker, args=(r, world, port, path, ask, q)) for r in range(world)]
    [p.start() for p in procs]
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda t: t[0])
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    for rank, got in res:
        assert got == want, rank


# ---- 4. the carry by hand: two GpuIndex shards ---------------------------------------------------------------------
def _lists(ix):
    """(term_offsets, doc_ids) of an index's BM25 part, finalized or not"""
    to = np.empty(ix.n_terms + 1, dtype=np.uint64)
    di = np.empty(int(ix.bm25_local_stats()[2]), dtype=np.uint32)
    ix._ck(ix.L.oi_index_read_bm25(ix.h, to.ctypes.data, di.ctypes.data, None, None, None))
    return to.astype(np.int64), di.astype(np.int64)


def _shard_pair(oi, texts, sources, cut):
    from openintel_b200 import capi
    with capi.GpuLexicon() as lx:
        pol, spec, _, _ = lx.analyze(texts)
    src = np.array([0 if s == "reddit" else 1 for s in sources], dtype=np.uint8)
    full = oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1)
    vocab = full.build_bm25_text(texts)
    full.load_post_signals(pol, spec, src)
    parts = []
    for lo, hi in ((0, cut), (cut, len(texts))):
        ix = oi.GpuIndex(n_docs=hi - lo, dim=4, doc_base=lo, max_k=1)
        parts.append((ix, ix.build_bm25_text(texts[lo:hi])))
        ix.load_post_signals(pol[lo:hi], spec[lo:hi], src[lo:hi])
    blob, offs = capi.pack_texts([w for _, v in parts for w in v])
    for ix, _ in parts:
        assert ix.bm25_union_vocabulary(blob, offs) == vocab
    return full, [ix for ix, _ in parts], vocab, pol, spec


def test_carry_continues_the_chain_across_two_shards(oi):
    texts, sources, tickers = _synthetic(20_000, 99, n_tickers=50)
    cut = 12_345
    full, (a, b), vocab, pol, spec = _shard_pair(oi, texts, sources, cut)
    ids = [vocab.index(t) for t in tickers[:30] if t in vocab] + [vocab.index("calls")]
    for src in (None, 0, 1):
        s_all, m_all = full.mention_summary(ids, source=src)
        s_a, m_a = a.mention_summary(ids, source=src)
        s_b, m_b = b.mention_summary(ids, source=src, carry=s_a)
        assert s_b.tobytes() == s_all.tobytes()
        for x, y in zip(m_b, m_all):
            _same_summary(x, y)
        # the first shard's summary is the summary of the prefix
        srcs = np.array([0 if s == "reddit" else 1 for s in sources])
        to, di = _lists(full)
        for i, t in enumerate(ids):
            d = di[to[t]:to[t + 1]]
            d = d[d < cut]
            if src is not None:
                d = d[srcs[d] == src]
            _same_summary(m_a[i], O.social_summary(pol[d], spec[d].astype(np.int32)), (t, src))
    for ix in (full, a, b):
        ix.close()


# ---- 5. errors and state --------------------------------------------------------------------------------------------
def test_errors_and_state(oi):
    texts = ["$GME to the moon", "gme puts", "calls on AMC", "nothing here", "GME GME dump", "amc squeeze yolo"]
    pol = np.array([O.lexicon_score(t)[0] for t in texts])
    spec = np.array([O.lexicon_score(t)[1] for t in texts], dtype=np.uint8)
    src = np.array([0, 1, 0, 1, 1, 0], dtype=np.uint8)
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        with pytest.raises(oi.OiError) as e:  # no BM25 part (and no signals)
            ix.mention_summary([0])
        assert e.value.status == 5
        ix.load_post_signals(pol, spec, src)
        with pytest.raises(oi.OiError) as e:  # signals, still no BM25 part
            ix.mention_summary([0])
        assert e.value.status == 5
    with oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1) as ix:
        vocab = ix.build_bm25_text(texts)
        with pytest.raises(oi.OiError) as e:  # a BM25 part, no signals
            ix.mention_summary([0])
        assert e.value.status == 5 and "signals" in e.value.message
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
    conn, mk = _fixture(G, db)
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
