"""`python -m openintel_b200.related` — what is being talked about together with a ticker, over a post store: per anchor
ticker, the terms its posts in a window [since, until) mention more often than independence predicts, ranked (SPEC §8d).
Each ranked term carries its co-mention count and the "social" block of the posts that mention both.

The co-mention counts of an anchor against every term come from one device call per shard and batch of anchors
(store.MentionIndex.comention_counts); rank() below is the §8d rule on the host:

    expected = (n_a * n_u) / N                       n_a, n_u: the anchor's and the term's posts in the window
    score    = (co - expected) / sqrt(expected + 1)  co: the posts in the window that mention both; N: all of them

    python -m openintel_b200.related --store posts.db --since 2024-01-08T00:00:00Z --until 2024-01-09T00:00:00Z \\
        [--top 20] [--min-co-mentions 1] [--source reddit] [--universe tickers.txt] GME AMC
"""
import argparse
import json
import sys

import numpy as np


def check_args(since, until, k, min_co_mentions):
    """the window and sizes of a ranking as ints, checked: since < until, k >= 1 and min_co_mentions >= 1"""
    since, until, k, min_co_mentions = int(since), int(until), int(k), int(min_co_mentions)
    if not since < until:
        raise ValueError("the window must satisfy since < until")
    if k < 1 or min_co_mentions < 1:
        raise ValueError("k and min_co_mentions must be at least 1")
    return since, until, k, min_co_mentions


def rank(co, n_u, n_a, n_posts, anchor, k, min_co_mentions=1, candidates=None):
    """The SPEC §8d ranking of one anchor.  co: co(anchor, u) per term u (term id = index); n_u: every term's mention
    count in the window; n_a = co(anchor, anchor); n_posts = N, the posts in the window; anchor: the anchor's term id,
    never ranked (None: no term is left out); candidates: a bool mask over the terms, or None for all.  A candidate has
    co >= min_co_mentions (and its mask bit).  An anchor with n_a = 0 ranks nothing.  IEEE f64, in exactly this
    association:
        expected = ((double)n_a * (double)n_u) / (double)N
        score    = ((double)co - expected) / sqrt(expected + 1.0)
    Order: score descending, ties by ascending term id; the first k.
    -> (term ids int64 [<= k], expected f64, score f64), in rank order"""
    co = np.asarray(co).reshape(-1)
    n_u = np.asarray(n_u).reshape(-1)
    n_a, n_posts, k, min_co_mentions = int(n_a), int(n_posts), int(k), int(min_co_mentions)
    if co.shape != n_u.shape:
        raise ValueError("co and n_u must have one count per term")
    if k < 1 or min_co_mentions < 1:
        raise ValueError("k and min_co_mentions must be at least 1")
    if n_a < 0 or n_posts < n_a:
        raise ValueError("need 0 <= n_a <= N, got n_a = %d, N = %d" % (n_a, n_posts))
    if n_a == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0), np.zeros(0)
    keep = co >= min_co_mentions
    if anchor is not None:
        keep[int(anchor)] = False
    if candidates is not None:
        keep &= np.asarray(candidates, dtype=bool).reshape(-1)
    ids = np.flatnonzero(keep)  # ascending term id
    expected = (np.float64(n_a) * n_u[ids].astype(np.float64)) / np.float64(n_posts)
    score = (co[ids].astype(np.float64) - expected) / np.sqrt(expected + 1.0)
    order = np.argsort(-score, kind="stable")[:k]  # stable: equal scores keep ascending term id
    return ids[order].astype(np.int64), expected[order], score[order]


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m openintel_b200.related",
                                 description="terms mentioned together with tickers more often than chance, in a window "
                                             "(one GPU call per 64 tickers)")
    ap.add_argument("--store", required=True, help="SQLite post store (openintel_b200.store schema)")
    ap.add_argument("--since", required=True, help="start of the window, RFC 3339 (e.g. 2024-01-08T00:00:00Z)")
    ap.add_argument("--until", required=True, help="end of the window, RFC 3339")
    ap.add_argument("--top", type=int, default=20, help="how many related terms to list per ticker (default 20)")
    ap.add_argument("--min-co-mentions", type=int, default=1,
                    help="least posts mentioning both the ticker and the term to be ranked (default 1)")
    ap.add_argument("--source", choices=["reddit", "bluesky"], help="only this source's posts")
    ap.add_argument("--universe", help="file of terms to rank among (whitespace-separated, '#' comments); default all")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("tickers", nargs="+", metavar="TICKER", help="anchor cashtags / words, e.g. GME or $GME")
    args = ap.parse_args(argv)
    from . import capi, store, timeline, trending
    try:
        since, until = (store.parse_created_at(x) for x in (args.since, args.until))
    except ValueError as e:
        ap.error(str(e))
    if not since < until:
        ap.error("--since must be before --until")
    if args.top < 1:
        ap.error("--top must be at least 1")
    if args.min_co_mentions < 1:
        ap.error("--min-co-mentions must be at least 1")
    universe = None
    if args.universe is not None:
        try:
            universe = trending.read_universe(args.universe)
        except (OSError, UnicodeDecodeError) as e:
            ap.error("--universe: %s" % e)
    conn = store.open_store(args.store)
    try:
        with store.MentionIndex(conn, device_index=args.device) as mi:
            anchors = mi.related(args.tickers, since, until, args.top, min_co_mentions=args.min_co_mentions,
                                 source=args.source, universe=universe)
    except (capi.OiError, ValueError) as e:  # a store without a token, a created_at without an offset
        sys.stderr.write("error: %s\n" % e)
        return 1
    finally:
        conn.close()
    out = {"since": timeline.format_time(since), "until": timeline.format_time(until), "source": args.source,
           "top": args.top, "min_co_mentions": args.min_co_mentions, "universe": args.universe, "anchors": anchors}
    sys.stdout.write(json.dumps(out) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
