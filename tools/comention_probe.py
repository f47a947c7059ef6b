#!/usr/bin/env python3
"""Cost of co-mention counts and shared-post summaries over the whole vocabulary (oi_index_comention_counts and
oi_index_comention_summary, SPEC §8d) next to the host path they replace: tokenize every post of the window and count
the tokens of the posts that hold an anchor (set intersection).

Corpus: the 2M-post corpus of tools/mention_summary_probe.py (seed 11) with the creation times of
tools/mention_counts_probe.py (uniform over 90 days, seed 12).  Anchors: the head ticker alone, the 8 and the 64 most
frequent tickers (the head ticker first).  Windows: one day in the middle of the span, and all 90 days.  Per (anchors,
window):
  * counts_call_ms: wall clock of the blocking call (the copy of n_anchors x n_terms u32 to the host included), the mean
    over --reps calls after two warm-up calls; counts_kernel_ms / mark_kernel_ms: the kernels from torch.profiler in a
    separate call; all_kernels_ms: every kernel of that call (the memsets and copies are in the call time only),
  * co_postings: the sum of the counts (the postings whose post carries an anchor), host_equal: the counts equal the
    host path's,
  * self_equal: co(a, a) equals oi_index_mention_counts over [since, until),
  * pairs: the summaries of (anchor, its 20 most co-mentioned terms) for every anchor in one call -- pairs_call_ms as
    above, pairs_kernel_ms (every kernel), and pair_self_equal: pair(a, a) equals oi_index_mention_timeline's one-bucket
    state bit for bit.
host_path_s: the host path for the 64 anchors (one pass: tokenize + intersect), per window.  The card name and power
limit are read in the same run.  Prints one JSON line."""
import argparse
import collections
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--posts", type=int, default=2_000_000)
    ap.add_argument("--words", type=int, default=1_000_000)
    ap.add_argument("--tickers", type=int, default=2000)
    ap.add_argument("--days", type=int, default=90)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    import torch  # noqa: F401  (CUDA context for the profiler)
    import openintel_b200 as oi
    from openintel_b200 import analyze, capi, hostlib
    from mention_summary_probe import mention_corpus
    from mention_timeline_probe import profile_kernels
    from text_index_probe import gpu_info

    gpu = gpu_info()
    t0 = time.perf_counter()
    texts, tickers, src = mention_corpus(a.posts, a.words, a.tickers, 11)
    times = T0 + np.random.default_rng(12).integers(0, a.days * DAY, len(texts))
    gen_s = time.perf_counter() - t0
    ix = oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1)
    vocab = ix.build_bm25_text(texts)
    V = len(vocab)
    tid = {w: i for i, w in enumerate(vocab)}
    with capi.GpuLexicon(reserve_bytes=1 << 28, reserve_posts=len(texts)) as lx:
        pol, spec, _, _ = lx.analyze(texts)
    ix.load_post_signals(pol, spec, src)
    ix.load_post_times(times)
    n_post = int(ix.bm25_local_stats()[2])
    known = [analyze.ticker_key(t) for t in tickers if analyze.ticker_key(t) in tid]
    all_counts = ix.mention_counts([T0, T0 + a.days * DAY])[:, 0]
    order = sorted(known[1:], key=lambda t: -int(all_counts[tid[t]]))
    sets = {1: [known[0]], 8: [known[0]] + order[:7], 64: [known[0]] + order[:63]}
    mid = T0 + (a.days // 2) * DAY
    windows = {"1d": [mid, mid + DAY], "90d": [T0, T0 + a.days * DAY]}

    res, host = {}, {}
    for wname, w in windows.items():
        # the host path for the 64 anchors: tokenize every post of the window, count the tokens of the anchors' posts
        anchors = sets[64]
        t0 = time.perf_counter()
        cnt = {x: collections.Counter() for x in anchors}
        for d, t in enumerate(texts):
            if w[0] <= times[d] < w[1]:
                toks = set(hostlib.tokenize(t))
                for x in toks.intersection(anchors):
                    cnt[x].update(toks)
        host[wname] = round(time.perf_counter() - t0, 2)
        want = np.zeros((len(anchors), V), dtype=np.int64)
        for i, x in enumerate(anchors):
            for u, c in cnt[x].items():
                want[i, tid[u]] = c
        rows = {x: want[i] for i, x in enumerate(anchors)}
        n_u = ix.mention_counts(w)[:, 0]
        for na, names in sets.items():
            ids = np.array([tid[x] for x in names], dtype=np.uint32)
            e = np.array(w, dtype=np.int64)

            def call():
                return ix.comention_counts(ids, e)
            call()
            out = call()
            t0 = time.perf_counter()
            for _ in range(a.reps):
                call()
            call_ms = (time.perf_counter() - t0) / a.reps * 1e3
            ks = profile_kernels(call)
            # the pairs: every anchor with its 20 most co-mentioned other terms, and itself
            pa, pu = [], []
            for i, x in enumerate(ids):
                row = out[i].astype(np.int64)
                row[x] = -1
                top = np.argsort(-row, kind="stable")[:20]
                pa += [int(x)] * 21
                pu += [int(x)] + [int(u) for u in top]
            pa, pu = np.array(pa, dtype=np.uint32), np.array(pu, dtype=np.uint32)

            def pairs():
                return ix.comention_summary(pa, pu, e)
            pairs()
            st, _ = pairs()
            t0 = time.perf_counter()
            for _ in range(a.reps):
                pairs()
            pairs_ms = (time.perf_counter() - t0) / a.reps * 1e3
            pks = profile_kernels(pairs)
            tl, _ = ix.mention_timeline(ids, e)
            self_rows = st[np.arange(len(ids)) * 21]
            r = {"anchors": int(na), "window_s": int(w[1] - w[0]), "terms": V, "postings": n_post,
                 "counts_call_ms": round(call_ms, 3),
                 "counts_kernel_ms": round(sum(v for k, v in ks.items() if "comention_counts_kernel" in k), 3),
                 "mark_kernel_ms": round(sum(v for k, v in ks.items() if "comention_mark_kernel" in k), 3),
                 "all_kernels_ms": round(sum(ks.values()), 3), "co_postings": int(out.sum(dtype=np.int64)),
                 "host_equal": bool(all((out[i] == rows[x]).all() for i, x in enumerate(names))),
                 "self_equal": bool((out[np.arange(len(ids)), ids] == n_u[ids]).all()),
                 "pairs": int(len(pa)), "pair_posts": int(st["total"].sum()), "pairs_call_ms": round(pairs_ms, 3),
                 "pairs_kernel_ms": round(sum(pks.values()), 3),
                 "pair_self_equal": self_rows.tobytes() == tl[:, 0].tobytes()}
            res["%s_A%d" % (wname, na)] = r
            print(wname, na, json.dumps(r), file=sys.stderr, flush=True)
    ix.close()
    print(json.dumps({
        "workload": "oi_index_comention_counts / _summary: %d posts over %d days, %d terms, %d postings" % (len(texts), a.days, V,
                                                                                                          n_post),
        "gpu": gpu, "corpus_gen_s": round(gen_s, 1), "reps": a.reps, "runs": res, "host_path_s_64_anchors": host,
        "head_ticker": known[0], "head_posts": int(all_counts[tid[known[0]]])}), flush=True)


if __name__ == "__main__":
    main()
