#!/usr/bin/env python3
"""Cost of per-ticker timelines from the index (oi_index_mention_timeline, SPEC §8b) next to the `analyze --mention
--since --until` host path on the same posts, with every (ticker, bucket) summary checked against the oracle.

Corpus: the 2M-post corpus of tools/mention_summary_probe.py (2000 Zipf-distributed tickers, a head ticker in ~30 % of
the posts), with random creation times over 90 days, not monotonic in doc id.  Layouts: the 1000 most frequent
tickers at daily (B = 90) and hourly (B = 2160) buckets, the head ticker alone at B = 1 and B = 90.  Per layout:
  * call_ms: wall clock of the blocking call (best of the reps),
  * kernel_ms: all kernels of one call from torch.profiler in a separate call, split into keys_sort_offsets_ms (lengths,
    scan, keys, radix sort, segment offsets) and summaries_ms (mention_timeline_kernel),
  * segments / postings / longest_chain: (term, bucket) segments, requested postings, and the most posts with a non-zero
    polarity in one segment (the longest dependent DADD chain),
  * oracle_equal: every (ticker, bucket) summary equals oracle.social_summary over the posts of the ticker in the bucket.
host_path_s: analyze.select_posts(mention, since, until) + GpuLexicon per (ticker, bucket) on a sample, over a SQLite
store of the same posts.  The card name and power limit are read in the same run.  Prints one JSON line."""
import argparse
import ctypes as C
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

T0 = 1704067200  # 2024-01-01T00:00:00Z
DAY = 86400


def profile_kernels(fn):
    """{kernel name: ms} of one run of fn"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    out = {}
    for e in prof.key_averages():
        dt = getattr(e, "self_device_time_total", None)
        dt = dt if dt is not None else getattr(e, "self_cuda_time_total", 0.0)
        if dt and "Memcpy" not in e.key and "Memset" not in e.key:
            out[e.key] = out.get(e.key, 0.0) + dt / 1e3
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--posts", type=int, default=2_000_000)
    ap.add_argument("--words", type=int, default=1_000_000)
    ap.add_argument("--tickers", type=int, default=2000)
    ap.add_argument("--batch", type=int, default=1000)
    ap.add_argument("--days", type=int, default=90)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch  # noqa: F401  (CUDA context for the profiler)
    import oracle as O
    import openintel_b200 as oi
    from openintel_b200 import analyze, capi, store, timeline
    from mention_summary_probe import mention_corpus
    from text_index_probe import gpu_info

    t0 = time.perf_counter()
    texts, tickers, src = mention_corpus(a.posts, a.words, a.tickers, 11)
    times = T0 + np.random.default_rng(12).integers(0, a.days * DAY, len(texts))
    gen_s = time.perf_counter() - t0
    ix = oi.GpuIndex(n_docs=len(texts), dim=4, max_k=1)
    vocab = ix.build_bm25_text(texts)
    term_id = {w: i for i, w in enumerate(vocab)}
    with capi.GpuLexicon(reserve_bytes=1 << 28, reserve_posts=len(texts)) as lx:
        pol, spec, _, _ = lx.analyze(texts)
    ix.load_post_signals(pol, spec, src)
    t0 = time.perf_counter()
    ix.load_post_times(times)
    load_times_ms = (time.perf_counter() - t0) * 1e3

    to = np.empty(ix.n_terms + 1, dtype=np.uint64)
    doc_ids = np.empty(int(ix.bm25_local_stats()[2]), dtype=np.uint32)
    ix._ck(ix.L.oi_index_read_bm25(ix.h, to.ctypes.data, doc_ids.ctypes.data, None, None, None))
    to, doc_ids = to.astype(np.int64), doc_ids.astype(np.int64)
    lens = {w: int(to[term_id[w] + 1] - to[term_id[w]]) for w in tickers if w in term_id}
    batch = sorted(lens, key=lambda w: -lens[w])[:a.batch]
    ids = np.array([term_id[w] for w in batch], dtype=np.uint32)
    daily = T0 + DAY * np.arange(a.days + 1, dtype=np.int64)
    hourly = T0 + 3600 * np.arange(24 * a.days + 1, dtype=np.int64)
    layouts = {"batch_daily": (ids, daily), "batch_hourly": (ids, hourly), "head_B1": (ids[:1], daily[[0, -1]]),
               "head_daily": (ids[:1], daily)}

    opol = np.empty(len(texts))
    ospec = np.empty(len(texts), dtype=np.int32)
    for d, t in enumerate(texts):
        opol[d], ospec[d] = O.lexicon_score(t)[:2]
    empty = O.social_summary(opol[:0], ospec[:0])

    def same(sm, o):
        return all(struct.pack("<d", float(sm[f])) == struct.pack("<d", float(o[f])) for f in o)

    res, ok = {}, True
    for name, (tids, edges) in layouts.items():
        n, nb = len(tids), len(edges) - 1
        states = np.zeros(n * nb, dtype=capi.MENTION_STATE_DTYPE)
        sums = np.zeros(n * nb, dtype=capi.SOCIAL_SUMMARY_DTYPE)

        def call():
            ix._ck(ix.L.oi_index_mention_timeline(ix.h, tids.ctypes.data, n, edges.ctypes.data, nb, -1, C.c_double(0.2), None,
                                                  states.ctypes.data, sums.ctypes.data))
        call()
        ts = []
        for _ in range(a.reps):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        ks = profile_kernels(call)
        summ = sum(v for k, v in ks.items() if "mention_timeline_kernel" in k)
        # the check: per ticker, its posts split by bucket in doc order, against the oracle
        sm = capi.summaries_from_array(sums)
        longest, postings = 0, 0
        for i, t in enumerate(tids):
            d = doc_ids[to[t]:to[t + 1]]
            postings += len(d)
            b = np.searchsorted(edges, times[d], side="right") - 1
            order = np.argsort(b, kind="stable")
            cuts = np.searchsorted(b[order], np.arange(nb + 1))
            for k in range(nb):
                dk = d[order[cuts[k]:cuts[k + 1]]]
                if len(dk):
                    ok &= same(sm[i * nb + k], O.social_summary(opol[dk], ospec[dk]))
                    longest = max(longest, int(np.count_nonzero(opol[dk])))
                else:
                    ok &= same(sm[i * nb + k], empty)
        res[name] = {"tickers": n, "buckets": nb, "segments": n * nb, "postings": postings, "longest_chain": longest,
                     "call_ms": round(min(ts) * 1e3, 3), "kernel_ms": round(sum(ks.values()), 3),
                     "keys_sort_offsets_ms": round(sum(ks.values()) - summ, 3), "summaries_ms": round(summ, 3)}
        print(name, json.dumps(res[name]), file=sys.stderr, flush=True)
    # B = 1 around all posts is the whole-list summary
    ok &= ix.mention_timeline(ids, daily[[0, -1]])[0][:, 0].tobytes() == ix.mention_summary(ids)[0].tobytes()

    # the host path on a sample of (ticker, bucket) pairs
    host = []
    with tempfile.TemporaryDirectory() as tmp:
        conn = store.open_store(os.path.join(tmp, "posts.db"))
        store.insert_posts(conn, [dict(id="p%d" % i, source=store.SOURCES[src[i]], author="a", text=t,
                                       created_at=timeline.format_time(int(times[i])), engagement=0) for i, t in enumerate(texts)])
        with capi.GpuLexicon() as lx:
            for w, k in ((batch[0], 10), (batch[len(batch) // 2], 40), (batch[-1], 80)):
                t0 = time.perf_counter()
                _, s_w, t_w = analyze.select_posts(conn, mention="$" + w.upper(), since=int(daily[k]), until=int(daily[k + 1]))
                if t_w:
                    analyze.analyze_posts(lx, s_w, t_w)
                host.append(dict(ticker=w, bucket=k, posts=len(t_w), s=round(time.perf_counter() - t0, 3)))
        conn.close()
    ix.close()
    print(json.dumps({
        "workload": "oi_index_mention_timeline: %d posts over %d days, %d terms; %d tickers asked; head ticker in %d posts" % (
            len(texts), a.days, len(vocab), len(batch), lens[batch[0]]),
        "gpu": gpu_info(), "corpus_gen_s": round(gen_s, 1), "load_times_ms": round(load_times_ms, 2),
        "layouts": res, "host_path_s_per_ticker_bucket": host, "oracle_equal": bool(ok)}), flush=True)


if __name__ == "__main__":
    main()
