"""Helpers shared by the GPU tests of the mention calls (SPEC §8a-c): the library fixture, the synthetic and reference
corpora and their stores, bitwise summary comparison, two-shard and sharded set-ups and the gloo rank harness."""
import json
import os
import socket
import struct

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T0 = 1704067200  # 2024-01-01T00:00:00Z
DAY = 86400
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


def iso(t):
    from openintel_b200 import timeline
    return timeline.format_time(int(t))


def bits(x):
    return struct.pack("<d", float(x))


def same_summary(a, b, what=""):
    for f in FIELDS:
        if isinstance(b[f], float):
            assert bits(a[f]) == bits(b[f]), (what, f, a[f], b[f])
        else:
            assert a[f] == b[f], (what, f, a[f], b[f])


def make_store(path, texts, sources, times=None):
    """a store WITHOUT embeddings (the mention path does not need them); times: created_at per post, seconds since the
    Unix epoch, or None for all at T0"""
    from openintel_b200 import store
    conn = store.open_store(path)
    store.insert_posts(conn, [dict(id="p%d" % i, source=s, author="a%d" % (i % 97), text=t,
                                   created_at=iso(T0 if times is None else times[i]), engagement=i % 50)
                              for i, (t, s) in enumerate(zip(texts, sources))])
    return conn


def fixture_store(G, path):
    """the reference fixture posts at distinct hourly times not in doc order -> (conn, mock market, hours)"""
    from openintel_b200 import fusion
    fx = G["fixture_posts"]["posts"]
    hours = np.random.default_rng(5).permutation(len(fx))
    conn = make_store(path, [p["text"] for p in fx], [p["source"] for p in fx], T0 + 3600 * hours)
    m = G["fixture_posts"]["mock_market"]
    return conn, fusion.MarketSummary.from_snapshot(m["last_price"], m["previous_close"], m["volume"], m["avg_volume"],
                                                    m["iv_rank"]), hours


# ---- the synthetic corpus -------------------------------------------------------------------------------------------
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


def synthetic(n_posts, seed, n_tickers=300):
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


# ---- the six-post corpus of the errors and state tests -----------------------------------------------------------
SMALL_TEXTS = ["$GME to the moon", "gme puts", "calls on AMC", "nothing here", "GME GME dump", "amc squeeze yolo"]
SMALL_EDGES = [T0, T0 + 24 * 3600, T0 + 48 * 3600]


def small_corpus():
    """-> (texts, polarity, speculative, source codes, times) of the six posts"""
    pol = np.array([O.lexicon_score(t)[0] for t in SMALL_TEXTS])
    spec = np.array([O.lexicon_score(t)[1] for t in SMALL_TEXTS], dtype=np.uint8)
    src = np.array([0, 1, 0, 1, 1, 0], dtype=np.uint8)
    times = T0 + np.array([50, 10, 20, 30, 40, 0]) * 3600
    return list(SMALL_TEXTS), pol, spec, src, times


# ---- shards -----------------------------------------------------------------------------------------------------------
def lists(ix):
    """(term_offsets, doc_ids) of an index's BM25 part, finalized or not"""
    to = np.empty(ix.n_terms + 1, dtype=np.uint64)
    di = np.empty(int(ix.bm25_local_stats()[2]), dtype=np.uint32)
    ix._ck(ix.L.oi_index_read_bm25(ix.h, to.ctypes.data, di.ctypes.data, None, None, None))
    return to.astype(np.int64), di.astype(np.int64)


def shard_pair(oi, texts, sources, cut):
    """the whole corpus and its two shards [0, cut) and [cut, n) as GpuIndex with signals, the shards over the united
    vocabulary -> (full, [a, b], vocab, polarity, speculative)"""
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


N_SHARD = 3000


def sharded_corpus(seed, world, tokenless):
    """the synthetic corpus of the sharded tests (N_SHARD posts, 60 tickers): `onlyfirst` appears on the first shard
    only; with `tokenless`, the middle shard's posts hold no token at all (its lists are all empty)"""
    from openintel_b200 import sharding
    texts, sources, tickers = synthetic(N_SHARD, seed, n_tickers=60)
    texts[3] += " onlyfirst moon"
    texts[10] += " onlyfirst dump"
    if tokenless:
        base, n = sharding.shard_range(N_SHARD, world, 1)
        for i in range(base, base + n):
            texts[i] = ("!!!", "ÿþ ???", "... — !!", "\U0001f680 $$")[i % 4]
    return texts, sources, tickers


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_main(rank, world, port, q, worker, args):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        q.put((rank, worker(dist, *args)))
    finally:
        dist.destroy_process_group()


def run_ranks(world, worker, *args):
    """runs worker(dist, *args) on `world` spawned gloo ranks (all on device 0) -> [(rank, its result)] in rank order;
    every rank must exit cleanly.  `worker` is a top-level function of a test module."""
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_rank_main, args=(r, world, port, q, worker, args)) for r in range(world)]
    [p.start() for p in procs]
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda t: t[0])
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    return res
