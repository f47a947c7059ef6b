"""`python -m openintel_b200.authors` — who talks about a ticker, over a post store: per ticker, its posts in a window
[since, until) grouped by author, the authors with the most posts, and how concentrated the talk is (SPEC §8e).  One
account posting 500 times and 500 accounts posting once each look alike to `compare`, `timeline` and `trending`; here
the first shows hhi = 1 and effective_authors = 1, the second effective_authors = 500.

The (ticker, author) runs of many tickers come from one device call per shard (store.MentionIndex.authors); merge()
and rank() below are the §8e rules on the host:

    P = sum of posts over the ticker's authors, A = their number, S = sum of posts^2 (an exact integer)
    hhi               = S / (P * P)
    effective_authors = (P * P) / S
    top_share         = (posts of the first k ranked authors) / P

    python -m openintel_b200.authors --store posts.db --since 2024-01-08T00:00:00Z --until 2024-01-09T00:00:00Z \\
        [--top 10] [--source reddit] GME AMC
"""
import argparse
import json
import sys

import numpy as np

from . import capi

_U64_MAX = np.uint64(0xFFFFFFFFFFFFFFFF)
_SUMMED = ("posts", "bullish", "bearish", "speculative", "engagement")


def check_args(since, until, k):
    """the window and size of a ranking as ints, checked: since < until and k >= 1"""
    since, until, k = int(since), int(until), int(k)
    if not since < until:
        raise ValueError("the window must satisfy since < until")
    if k < 1:
        raise ValueError("k must be at least 1")
    return since, until, k


def merge(runs_per_rank):
    """The SPEC §8e merge of the shards' runs (capi.AUTHOR_RUN_DTYPE each, any order): one run per (term, author), the
    counts and engagement summed, first_at the min and last_at the max.  Integers only, so the result does not depend
    on the order of the shards.  -> AUTHOR_RUN_DTYPE sorted by (term, author)"""
    runs = np.concatenate([np.asarray(r, dtype=capi.AUTHOR_RUN_DTYPE).reshape(-1) for r in runs_per_rank] or
                          [np.zeros(0, dtype=capi.AUTHOR_RUN_DTYPE)])
    runs = runs[np.lexsort((runs["author"], runs["term"]))]
    if not len(runs):
        return runs
    head = np.ones(len(runs), dtype=bool)
    head[1:] = (runs["term"][1:] != runs["term"][:-1]) | (runs["author"][1:] != runs["author"][:-1])
    starts = np.flatnonzero(head)
    out = runs[starts].copy()
    for f in _SUMMED:
        out[f] = np.add.reduceat(runs[f], starts)
    out["first_at"] = np.minimum.reduceat(runs["first_at"], starts)
    out["last_at"] = np.maximum.reduceat(runs["last_at"], starts)
    return out


def rank(runs, k):
    """The SPEC §8e figures and order of one term's runs (capi.AUTHOR_RUN_DTYPE, one per author).  IEEE f64, in exactly
    this association, with P = sum of posts, S = sum of posts^2 (exact):
        hhi               = (double)S / ((double)P * (double)P)
        effective_authors = ((double)P * (double)P) / (double)S
        top_share         = (double)(posts of the first k) / (double)P
    Order: posts descending, then engagement descending, then author id ascending; the first k.  P = 0: the figures are
    0 and nothing is ranked.  -> dict(mentions=P, authors, engagement, hhi, effective_authors, top_share, top: the first
    k runs in rank order)"""
    runs = np.asarray(runs, dtype=capi.AUTHOR_RUN_DTYPE).reshape(-1)
    k = int(k)
    if k < 1:
        raise ValueError("k must be at least 1")
    posts = runs["posts"].astype(np.uint64)
    P = int(posts.sum(dtype=np.uint64))
    out = dict(mentions=P, authors=int(len(runs)), engagement=int(runs["engagement"].sum(dtype=np.uint64)), hhi=0.0,
               effective_authors=0.0, top_share=0.0, top=runs[:0])
    if P == 0:
        return out
    S = int((posts * posts).sum(dtype=np.uint64))  # S <= P^2 < 2^64: exact
    order = np.lexsort((runs["author"], _U64_MAX - runs["engagement"].astype(np.uint64), _U64_MAX - posts))[:k]
    top = runs[order]
    pp = float(P) * float(P)
    out.update(hhi=float(S) / pp, effective_authors=pp / float(S), top_share=float(int(top["posts"].sum(dtype=np.uint64))) / float(P),
               top=top)
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m openintel_b200.authors",
                                 description="who posts about tickers in a window, and how concentrated the talk is "
                                             "(one GPU call for all tickers)")
    ap.add_argument("--store", required=True, help="SQLite post store (openintel_b200.store schema)")
    ap.add_argument("--since", required=True, help="start of the window, RFC 3339 (e.g. 2024-01-08T00:00:00Z)")
    ap.add_argument("--until", required=True, help="end of the window, RFC 3339")
    ap.add_argument("--top", type=int, default=10, help="how many authors to list per ticker (default 10)")
    ap.add_argument("--source", choices=["reddit", "bluesky"], help="only this source's posts")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("tickers", nargs="+", metavar="TICKER", help="cashtags / words, e.g. GME or $GME")
    args = ap.parse_args(argv)
    from . import store, timeline
    try:
        since, until = (store.parse_created_at(x) for x in (args.since, args.until))
    except ValueError as e:
        ap.error(str(e))
    if not since < until:
        ap.error("--since must be before --until")
    if args.top < 1:
        ap.error("--top must be at least 1")
    conn = store.open_store(args.store)
    try:
        with store.MentionIndex(conn, device_index=args.device) as mi:
            tickers = mi.authors(args.tickers, since, until, args.top, source=args.source)
    except (capi.OiError, ValueError) as e:  # a store without a token, a created_at without an offset
        sys.stderr.write("error: %s\n" % e)
        return 1
    finally:
        conn.close()
    out = {"since": timeline.format_time(since), "until": timeline.format_time(until), "source": args.source,
           "top": args.top, "tickers": tickers}
    sys.stdout.write(json.dumps(out) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
