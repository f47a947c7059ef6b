#!/usr/bin/env python3
"""Cost of per-term mention counts over the whole vocabulary (oi_index_mention_counts, SPEC §8c) next to the routes that
gave the same numbers before it: oi_index_mention_timeline over every term (its state's `total`), and a one-pass host
count (tokenize + Counter).  Then the wall time of store.MentionIndex.trending on a store of the same posts.

Corpus: the 2M-post corpus of tools/mention_summary_probe.py with the random creation times over 90 days of
tools/mention_timeline_probe.py.  Layouts: B = 2 (a 7-day baseline and a 1-day window, the trending call's edges) and
B = 90 (daily).  Per layout:
  * counts_call_ms: wall clock of the blocking call, best of the reps; counts_kernel_ms: its kernels from torch.profiler
    in a separate call (mention_counts_kernel; the memset and the copies are in the call time only),
  * B = 2 only: timeline_call_ms, the same counts through oi_index_mention_timeline over all terms (its states and
    summaries are 120 bytes per (term, bucket), 9 GB at B = 90, so that layout skips it), and timeline_equal,
  * oracle_equal: B = 2 against the host Counter; B = 90 against a numpy count over the CSR's doc ids and the times.
host_count_s: the one-pass host count at B = 2.  trending: MentionIndex over a SQLite store of the same posts -- the
lift, the first trending call (which parses and loads the post times) and the best of the later calls.  The card name
and power limit are read in the same run.  Prints one JSON line."""
import argparse
import ctypes as C
import collections
import json
import os
import sys
import tempfile
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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-store", action="store_true", help="skip the MentionIndex.trending part")
    a = ap.parse_args()
    import torch  # noqa: F401  (CUDA context for the profiler)
    import openintel_b200 as oi
    from openintel_b200 import capi, hostlib, store, timeline
    from mention_summary_probe import mention_corpus
    from mention_timeline_probe import profile_kernels
    from text_index_probe import gpu_info

    t0 = time.perf_counter()
    texts, tickers, src = mention_corpus(a.posts, a.words, a.tickers, 11)
    times = T0 + np.random.default_rng(12).integers(0, a.days * DAY, len(texts))
    gen_s = time.perf_counter() - t0
    ix = oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1)
    vocab = ix.build_bm25_text(texts)
    V = len(vocab)
    with capi.GpuLexicon(reserve_bytes=1 << 28, reserve_posts=len(texts)) as lx:
        pol, spec, _, _ = lx.analyze(texts)
    ix.load_post_signals(pol, spec, src)
    ix.load_post_times(times)
    to = np.empty(V + 1, dtype=np.uint64)
    n_post = int(ix.bm25_local_stats()[2])
    doc_ids = np.empty(n_post, dtype=np.uint32)
    ix._ck(ix.L.oi_index_read_bm25(ix.h, to.ctypes.data, doc_ids.ctypes.data, None, None, None))
    term_of = np.repeat(np.arange(V, dtype=np.int64), np.diff(to.astype(np.int64)))

    # the trending layout: a 7-day baseline before a 1-day window in the middle of the span
    t1 = T0 + (a.days // 2) * DAY
    layouts = {"B2": np.array([t1 - 7 * DAY, t1, t1 + DAY], dtype=np.int64),
               "B90": T0 + DAY * np.arange(a.days + 1, dtype=np.int64)}
    res, got = {}, {}
    for name, edges in layouts.items():
        nb = len(edges) - 1
        out = np.zeros((V, nb), dtype=np.uint32)

        def call():
            ix._ck(ix.L.oi_index_mention_counts(ix.h, edges.ctypes.data, nb, -1, out.ctypes.data))
        call()
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        ks = profile_kernels(call)
        got[name] = out.copy()
        b = np.searchsorted(edges, times[doc_ids], side="right") - 1
        keep = (b >= 0) & (b < nb)
        want = np.bincount(term_of[keep] * nb + b[keep], minlength=V * nb).reshape(V, nb)
        r = {"terms": V, "buckets": nb, "postings": n_post, "counted": int(keep.sum()), "counts_call_ms": round(min(ts) * 1e3, 3),
             "counts_kernel_ms": round(sum(v for k, v in ks.items() if "mention_counts_kernel" in k), 3),
             "all_kernels_ms": round(sum(ks.values()), 3), "csr_numpy_equal": bool((want == out).all())}
        if nb == 2:
            ids = np.arange(V, dtype=np.uint32)
            states = np.zeros(V * nb, dtype=capi.MENTION_STATE_DTYPE)
            sums = np.zeros(V * nb, dtype=capi.SOCIAL_SUMMARY_DTYPE)

            def tl():
                ix._ck(ix.L.oi_index_mention_timeline(ix.h, ids.ctypes.data, V, edges.ctypes.data, nb, -1, C.c_double(0.2), None,
                                                      states.ctypes.data, sums.ctypes.data))
            tl()
            ts = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                tl()
                ts.append(time.perf_counter() - t0)
            r["timeline_call_ms"] = round(min(ts) * 1e3, 3)
            r["timeline_kernel_ms"] = round(sum(profile_kernels(tl).values()), 3)
            r["timeline_equal"] = bool((states["total"].reshape(V, nb) == out).all())
            r["speedup_vs_timeline"] = round(r["timeline_call_ms"] / r["counts_call_ms"], 1)
        res[name] = r
        print(name, json.dumps(r), file=sys.stderr, flush=True)

    # the one-pass host count at B = 2: tokenize every post of the two windows, count (term, bucket)
    e2 = layouts["B2"]
    t0 = time.perf_counter()
    cnt = collections.Counter()
    for d, t in enumerate(texts):
        tt = times[d]
        if e2[0] <= tt < e2[2]:
            b = 0 if tt < e2[1] else 1
            cnt.update((w, b) for w in set(hostlib.tokenize(t)))
    host_s = time.perf_counter() - t0
    host = np.zeros((V, 2), dtype=np.int64)
    tid = {w: i for i, w in enumerate(vocab)}
    for (w, b), n in cnt.items():
        host[tid[w], b] = n
    res["B2"]["oracle_equal"] = bool((host == got["B2"]).all())
    res["B90"]["oracle_equal"] = res["B90"]["csr_numpy_equal"]
    ix.close()

    tr = None
    if not a.no_store:
        with tempfile.TemporaryDirectory() as tmp:
            conn = store.open_store(os.path.join(tmp, "posts.db"))
            store.insert_posts(conn, [dict(id="p%d" % i, source=store.SOURCES[src[i]], author="a", text=t,
                                           created_at=timeline.format_time(int(times[i])), engagement=0)
                                      for i, t in enumerate(texts)])
            t0 = time.perf_counter()
            mi = store.MentionIndex(conn)
            lift_s = time.perf_counter() - t0
            t0 = time.perf_counter()
            first = mi.trending(int(e2[1]), int(e2[2]), int(e2[0]), 20)
            first_s = time.perf_counter() - t0
            ts = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                ranked = mi.trending(int(e2[1]), int(e2[2]), int(e2[0]), 20)
                ts.append(time.perf_counter() - t0)
            c = mi.mention_counts(e2)
            tr = {"lift_s": round(lift_s, 2), "first_call_s": round(first_s, 3), "call_ms": round(min(ts) * 1e3, 2),
                  "counts_equal": bool((c == got["B2"]).all()), "same_list": ranked == first,
                  "top3": [(e["ticker"], e["mentions"], e["baseline_mentions"], round(e["surge"], 2)) for e in ranked[:3]]}
            mi.close()
            conn.close()
    print(json.dumps({
        "workload": "oi_index_mention_counts: %d posts over %d days, %d terms, %d postings" % (len(texts), a.days, V, n_post),
        "gpu": gpu_info(), "corpus_gen_s": round(gen_s, 1), "layouts": res, "host_count_s": round(host_s, 2),
        "trending": tr}), flush=True)


if __name__ == "__main__":
    main()
