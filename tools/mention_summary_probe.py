#!/usr/bin/env python3
"""Cost of per-ticker social summaries from the index (oi_index_mention_summary, SPEC §8a) next to the `analyze
--mention` host path on the same posts, with every summary checked against the oracle.

Corpus: the 2M-post Zipf corpus of tools/text_index_probe.py, with a pool of 2000 ticker tokens ($GME / Gme / gme,
Zipf-distributed, 0-2 per post), a head ticker in ~30 % of the posts and 0-3 lexicon words per post; random sources.
Prints one JSON line:
  * load_signals_ms: oi_index_load_post_signals (host check + copy of 2M signals), best of the reps,
  * batch_call_ms / batch_kernel_ms: one call for the 1000 most frequent tickers (wall clock of the blocking call, and
    the kernel alone from torch.profiler in a separate call),
  * head_call_ms / head_kernel_ms: one call for the head ticker alone,
  * ns_per_chained_post: head kernel time over the head list's posts with a non-zero polarity (the dependent DADD chain),
  * host_path_s_per_ticker: analyze.select_posts(mention=...) + GpuLexicon over a SQLite store of the same posts,
  * oracle_equal: all 1000 summaries (all posts and per source) equal oracle.social_summary over the posts that mention
    the ticker, bit for bit.
The card name and power limit are read in the same run."""
import argparse
import json
import os
import struct
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

LEX = ["moon", "calls", "long", "buy", "bullish", "squeeze", "breakout", "rocket", "pump", "rip", "green", "up", "rally",
       "bull", "puts", "short", "sell", "bearish", "dump", "crash", "drilling", "bagholder", "rug", "red", "down", "tank",
       "bear", "0dte", "yolo", "leaps", "theta", "gamma", "otm", "itm", "strike", "iv", "delta", "vega", "contracts"]


def mention_corpus(n_posts, n_words, n_tickers, seed):
    from text_index_probe import corpus
    texts, _ = corpus(n_posts, n_words, seed)
    rng = np.random.default_rng(seed + 1)
    tickers = ["tk%s" % np.base_repr(i, 36).lower() for i in range(n_tickers)]  # tickers[0] = the head ticker
    p = 1.0 / np.arange(1, n_tickers) ** 1.1
    n_tick, n_lex = rng.integers(0, 3, n_posts), rng.integers(0, 4, n_posts)
    tick = 1 + rng.choice(n_tickers - 1, size=int(n_tick.sum()), p=p / p.sum())
    lex = rng.integers(0, len(LEX), size=int(n_lex.sum()))
    head = rng.random(n_posts) < 0.3
    ti = li = 0
    out = []
    for i in range(n_posts):
        w = [("$" + tickers[t].upper(), tickers[t].capitalize(), tickers[t])[(i + j) % 3] for j, t in enumerate(tick[ti:ti + n_tick[i]])]
        ti += n_tick[i]
        w += [LEX[j] for j in lex[li:li + n_lex[i]]]
        li += n_lex[i]
        if head[i]:
            w.append("$" + tickers[0].upper())
        out.append(texts[i] + " " + " ".join(w) if w else texts[i])
    return out, tickers, rng.integers(0, 2, n_posts).astype(np.uint8)


def kernel_ms(fn, name):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    us = 0.0
    for e in prof.key_averages():
        if name in e.key:
            dt = getattr(e, "self_device_time_total", None)
            us += dt if dt is not None else getattr(e, "self_cuda_time_total", 0.0)
    return us / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--posts", type=int, default=2_000_000)
    ap.add_argument("--words", type=int, default=1_000_000)
    ap.add_argument("--tickers", type=int, default=2000)
    ap.add_argument("--batch", type=int, default=1000)
    ap.add_argument("--host-tickers", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch  # noqa: F401  (CUDA context for the profiler)
    import oracle as O
    import openintel_b200 as oi
    from openintel_b200 import analyze, capi, hostlib, store
    from text_index_probe import gpu_info

    t0 = time.perf_counter()
    texts, tickers, src = mention_corpus(a.posts, a.words, a.tickers, 11)
    gen_s = time.perf_counter() - t0
    ix = oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1)
    vocab = ix.build_bm25_text(texts)
    term_id = {w: i for i, w in enumerate(vocab)}
    with capi.GpuLexicon(reserve_bytes=1 << 28, reserve_posts=len(texts)) as lx:
        pol, spec, _, _ = lx.analyze(texts)

    def load():
        ix.load_post_signals(pol, spec, src)
    load()
    t_load = []
    for _ in range(a.reps):
        t0 = time.perf_counter()
        load()
        t_load.append(time.perf_counter() - t0)

    lens = {w: 0 for w in tickers}
    to = np.empty(ix.n_terms + 1, dtype=np.uint64)
    doc_ids = np.empty(int(ix.bm25_local_stats()[2]), dtype=np.uint32)
    ix._ck(ix.L.oi_index_read_bm25(ix.h, to.ctypes.data, doc_ids.ctypes.data, None, None, None))
    to, doc_ids = to.astype(np.int64), doc_ids.astype(np.int64)
    for w in tickers:
        if w in term_id:
            lens[w] = int(to[term_id[w] + 1] - to[term_id[w]])
    batch = sorted((w for w in tickers if lens[w]), key=lambda w: -lens[w])[:a.batch]
    ids = np.array([term_id[w] for w in batch], dtype=np.uint32)
    head_id = ids[:1]

    def timed(fn):
        fn()
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        return min(ts) * 1e3

    batch_ms = timed(lambda: ix.mention_summary(ids))
    head_ms = timed(lambda: ix.mention_summary(head_id))
    batch_k = kernel_ms(lambda: ix.mention_summary(ids), "mention_summary_kernel")
    head_k = kernel_ms(lambda: ix.mention_summary(head_id), "mention_summary_kernel")
    head_docs = doc_ids[to[head_id[0]]:to[head_id[0] + 1]]
    chained = int(np.count_nonzero(pol[head_docs]))
    longest = max(int(np.count_nonzero(pol[doc_ids[to[t]:to[t + 1]]])) for t in ids)

    # oracle: the posts whose tokens include the ticker (the rule of select_posts), the oracle's lexicon and summary
    t0 = time.perf_counter()
    want = set(batch)
    posts_of = {w: [] for w in batch}
    opol = np.empty(len(texts))
    ospec = np.empty(len(texts), dtype=np.int32)
    for d, t in enumerate(texts):
        for w in want.intersection(hostlib.tokenize(t)):
            posts_of[w].append(d)
        opol[d], ospec[d] = O.lexicon_score(t)[:2]
    ok = True
    for source in (None, 0, 1):
        states, sums = ix.mention_summary(ids, source=source)
        for i, w in enumerate(batch):
            d = np.array(posts_of[w], dtype=np.int64)
            if source is not None:
                d = d[src[d] == source]
            o = O.social_summary(opol[d], ospec[d])
            ok &= all(struct.pack("<d", float(sums[i][f])) == struct.pack("<d", float(o[f])) for f in o)
            ok &= [int(states[i]["by_source"][s]) for s in (0, 1)] == [int(np.sum(src[d] == s)) for s in (0, 1)]
    oracle_s = time.perf_counter() - t0

    # the host path: select_posts(mention=...) + GpuLexicon, per ticker, over a SQLite store of the same posts
    host = {}
    with tempfile.TemporaryDirectory() as tmp:
        conn = store.open_store(os.path.join(tmp, "posts.db"))
        store.insert_posts(conn, [dict(id="p%d" % i, source=store.SOURCES[src[i]], author="a", text=t,
                                       created_at="2024-01-01T00:00:00Z", engagement=0) for i, t in enumerate(texts)])
        pick = [batch[0], batch[len(batch) // 2], batch[-1]][:a.host_tickers]
        with capi.GpuLexicon() as lx:
            for w in pick:
                t0 = time.perf_counter()
                _, sources_w, texts_w = analyze.select_posts(conn, mention="$" + w.upper())
                rep, _, _ = analyze.analyze_posts(lx, sources_w, texts_w)
                host[w] = dict(posts=len(texts_w), s=round(time.perf_counter() - t0, 3))
                i = batch.index(w)
                ok &= rep["social"]["total_mentions"] == ix.mention_summary(ids[i:i + 1])[1][0]["total"]
        conn.close()
    ix.close()
    print(json.dumps({
        "workload": "oi_index_mention_summary: %d posts, %d terms, %d tickers asked, head ticker in %d posts (%d chained)" % (
            len(texts), len(vocab), len(batch), len(head_docs), chained),
        "gpu": gpu_info(), "corpus_gen_s": round(gen_s, 1),
        "load_signals_ms": round(min(t_load) * 1e3, 2),
        "batch_call_ms": round(batch_ms, 3), "batch_kernel_ms": round(batch_k, 3), "batch_longest_chain": longest,
        "head_call_ms": round(head_ms, 3), "head_kernel_ms": round(head_k, 3),
        "ns_per_chained_post": round(head_k * 1e6 / chained, 2) if chained else None,
        "host_path_s_per_ticker": host, "oracle_equal": bool(ok), "oracle_check_s": round(oracle_s, 1)}), flush=True)


if __name__ == "__main__":
    main()
