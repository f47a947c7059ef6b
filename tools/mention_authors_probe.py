#!/usr/bin/env python3
"""Cost of the per-author mention runs (oi_index_mention_authors, SPEC §8e) next to the host path they replace: tokenize
every post of the window and group the posts of the requested tickers by author.

Corpus: the 2M-post corpus of tools/mention_summary_probe.py (seed 11) with the creation times of
tools/mention_counts_probe.py (uniform over 90 days, seed 12).  Authors: --authors accounts, Zipf-distributed (exponent
1.1, seed 13), plus three planted accounts that post 20000 / 5000 / 1000 times about one ticker each (tickers 5, 6 and
7: the ticker is appended to the planted posts).  Engagement: uniform in [0, 1000).  Tickers: the head ticker alone,
and the 64 and the 1000 most frequent tickers (the head ticker first).  Windows: one day in the middle of the span,
and all 90 days.  Per (tickers, window):
  * call_ms: wall clock of the blocking call (the copy of the runs to the host included), the mean over --reps calls
    after two warm-up calls, with a capacity that fits; kernels_ms: every kernel of one call from torch.profiler in a
    separate call, aggregate_kernel_ms / keys_kernel_ms: the run-aggregation and the keys kernel alone,
  * postings: the postings of the requested lists, runs: the (ticker, author) runs, posts: their posts,
  * host_equal: the runs equal the host path's,
  * planted: for the set that holds tickers 5 to 7, each planted ticker's top author, its posts and its share.
host_path_s: the host path for the 1000 tickers (one pass: tokenize + group), per window.  The card name and power limit
are read in the same run.  Prints one JSON line."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

T0 = 1704067200  # 2024-01-01T00:00:00Z
DAY = 86400
PLANTED = ((5, 20000), (6, 5000), (7, 1000))  # (ticker index, posts) of the planted accounts


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--posts", type=int, default=2_000_000)
    ap.add_argument("--words", type=int, default=1_000_000)
    ap.add_argument("--tickers", type=int, default=2000)
    ap.add_argument("--authors", type=int, default=300_000)
    ap.add_argument("--days", type=int, default=90)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    import torch  # noqa: F401  (CUDA context for the profiler)
    import openintel_b200 as oi
    from openintel_b200 import analyze, authors, capi, hostlib
    from mention_summary_probe import mention_corpus
    from mention_timeline_probe import profile_kernels
    from text_index_probe import gpu_info

    gpu = gpu_info()
    t0 = time.perf_counter()
    texts, tickers, src = mention_corpus(a.posts, a.words, a.tickers, 11)
    times = T0 + np.random.default_rng(12).integers(0, a.days * DAY, len(texts))
    rng = np.random.default_rng(13)
    p = 1.0 / np.arange(1, a.authors + 1) ** 1.1
    author = rng.choice(a.authors, size=len(texts), p=p / p.sum()).astype(np.uint32)
    engagement = rng.integers(0, 1000, len(texts)).astype(np.uint32)
    taken = np.zeros(len(texts), dtype=bool)
    for j, (t, n) in enumerate(PLANTED):
        docs = rng.choice(np.flatnonzero(~taken), size=n, replace=False)
        taken[docs] = True
        author[docs] = a.authors + j
        for d in docs:
            texts[d] += " $" + tickers[t].upper()
    gen_s = time.perf_counter() - t0
    ix = oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1)
    vocab = ix.build_bm25_text(texts)
    tid = {w: i for i, w in enumerate(vocab)}
    with capi.GpuLexicon(reserve_bytes=1 << 28, reserve_posts=len(texts)) as lx:
        pol, spec, _, _ = lx.analyze(texts)
    ix.load_post_signals(pol, spec, src)
    ix.load_post_times(times)
    ix.load_post_authors(author, engagement)
    n_post = int(ix.bm25_local_stats()[2])
    known = [analyze.ticker_key(t) for t in tickers if analyze.ticker_key(t) in tid]
    all_counts = ix.mention_counts([T0, T0 + a.days * DAY])[:, 0]
    order = sorted(known[1:], key=lambda t: -int(all_counts[tid[t]]))
    sets = {1: [known[0]], 64: [known[0]] + order[:63], 1000: [known[0]] + order[:999]}
    mid = T0 + (a.days // 2) * DAY
    windows = {"1d": [mid, mid + DAY], "90d": [T0, T0 + a.days * DAY]}

    res, host = {}, {}
    for wname, w in windows.items():
        # the host path for the 1000 tickers: tokenize every post of the window, group the tickers' posts by author
        want_set = set(sets[1000])
        t0 = time.perf_counter()
        runs_h = {}
        for d in np.flatnonzero((times >= w[0]) & (times < w[1])):
            for t in want_set.intersection(hostlib.tokenize(texts[d])):
                r = runs_h.get((t, int(author[d])))
                x, tm = float(pol[d]), int(times[d])
                if r is None:
                    runs_h[(t, int(author[d]))] = [1, int(x > 0.2), int(x < -0.2), int(spec[d]), int(engagement[d]), tm, tm]
                else:
                    r[0] += 1
                    r[1] += x > 0.2
                    r[2] += x < -0.2
                    r[3] += int(spec[d])
                    r[4] += int(engagement[d])
                    r[5], r[6] = min(r[5], tm), max(r[6], tm)
        host[wname] = round(time.perf_counter() - t0, 2)
        for nt, names in sets.items():
            ids = np.array([tid[x] for x in names], dtype=np.uint32)
            e = np.array(w, dtype=np.int64)
            _, runs = ix.mention_authors(ids, e, capacity=1)  # sizes the buffer from the refusal
            cap = len(runs)

            def call():
                return ix.mention_authors(ids, e, capacity=cap)
            call()
            term_runs, runs = call()
            t0 = time.perf_counter()
            for _ in range(a.reps):
                call()
            call_ms = (time.perf_counter() - t0) / a.reps * 1e3
            ks = profile_kernels(call)
            got = {(names[int(r["term"])], int(r["author"])): [int(r[f]) for f in ("posts", "bullish", "bearish", "speculative",
                                                                                  "engagement", "first_at", "last_at")]
                   for r in runs}
            want = {k: [int(v) for v in r] for k, r in runs_h.items() if k[0] in set(names)}
            r = {"tickers": nt, "window_s": int(w[1] - w[0]), "postings": int(all_counts[ids].sum(dtype=np.int64)),
                 "runs": int(len(runs)), "posts": int(runs["posts"].sum()), "call_ms": round(call_ms, 3),
                 "kernels_ms": round(sum(ks.values()), 3),
                 "aggregate_kernel_ms": round(sum(v for k, v in ks.items() if "author_aggregate_kernel" in k), 3),
                 "keys_kernel_ms": round(sum(v for k, v in ks.items() if "author_keys_kernel" in k), 3),
                 "host_equal": got == want}
            planted = [tickers[t] for t, _ in PLANTED if tickers[t] in set(names)]
            if planted:
                r["planted"] = {}
                for x in planted:
                    i = names.index(x)
                    fig = authors.rank(runs[int(term_runs[i]):int(term_runs[i + 1])], 1)
                    top = fig["top"][0] if len(fig["top"]) else None
                    r["planted"][x] = {"top_author": None if top is None else int(top["author"]),
                                       "top_posts": None if top is None else int(top["posts"]),
                                       "top_share": fig["top_share"], "effective_authors": fig["effective_authors"],
                                       "authors": fig["authors"]}
            res["%s_T%d" % (wname, nt)] = r
            print(wname, nt, json.dumps(r), file=sys.stderr, flush=True)
    ix.close()
    print(json.dumps({
        "workload": "oi_index_mention_authors: %d posts over %d days, %d terms, %d postings, %d + %d authors" % (
            len(texts), a.days, len(vocab), n_post, a.authors, len(PLANTED)),
        "gpu": gpu, "corpus_gen_s": round(gen_s, 1), "reps": a.reps, "runs": res, "host_path_s_1000_tickers": host,
        "head_ticker": known[0], "head_posts": int(all_counts[tid[known[0]]])}), flush=True)


if __name__ == "__main__":
    main()
