"""`python -m openintel_b200.trending` — which tickers are suddenly being talked about, over a post store: every term of
the index ranked by how far its mention count in a window [since, until) rises above what a baseline window
[baseline-since, since) predicts (SPEC §8c).  Each ranked term carries the "social" block of `analyze --mention T` for
the baseline and for the window.

The counts of all terms come from one device call per shard (store.MentionIndex.mention_counts); rank() below is the
§8c rule on the host:

    expected = (m * (t2 - t1)) / (t1 - t0)          m: mentions in the baseline [t0, t1)
    surge    = (c - expected) / sqrt(expected + 1)  c: mentions in the window [t1, t2)

    python -m openintel_b200.trending --store posts.db --baseline-since 2024-01-01T00:00:00Z \\
        --since 2024-01-08T00:00:00Z --until 2024-01-09T00:00:00Z [--top 20] [--min-mentions 1] [--source reddit] \\
        [--universe tickers.txt]
"""
import argparse
import json
import sys

import numpy as np


def check_args(t0, t1, t2, k, min_mentions):
    """the times and sizes of a ranking as ints, checked: t0 < t1 < t2, k >= 1 and min_mentions >= 1"""
    t0, t1, t2, k, min_mentions = int(t0), int(t1), int(t2), int(k), int(min_mentions)
    if not t0 < t1 < t2:
        raise ValueError("the times must satisfy baseline_since < since < until")
    if k < 1 or min_mentions < 1:
        raise ValueError("k and min_mentions must be at least 1")
    return t0, t1, t2, k, min_mentions


def rank(c, m, t0, t1, t2, k, min_mentions=1, candidates=None):
    """The SPEC §8c ranking.  c / m: per-term mention counts in the window [t1, t2) and in the baseline [t0, t1), term
    id = index; candidates: a bool mask over the terms, or None for all.  A candidate has c >= min_mentions (and its
    mask bit).  IEEE f64, in exactly this association:
        expected = ((double)m * (double)(t2 - t1)) / (double)(t1 - t0)
        surge    = ((double)c - expected) / sqrt(expected + 1.0)
    Order: surge descending, ties by ascending term id; the first k.
    -> (term ids int64 [<= k], expected f64, surge f64), in rank order"""
    t0, t1, t2, k, min_mentions = check_args(t0, t1, t2, k, min_mentions)
    c = np.asarray(c).reshape(-1)
    m = np.asarray(m).reshape(-1)
    if c.shape != m.shape:
        raise ValueError("c and m must have one count per term")
    keep = c >= min_mentions
    if candidates is not None:
        keep &= np.asarray(candidates, dtype=bool).reshape(-1)
    ids = np.flatnonzero(keep)  # ascending term id
    cc, mm = c[ids].astype(np.float64), m[ids].astype(np.float64)
    expected = (mm * np.float64(t2 - t1)) / np.float64(t1 - t0)
    surge = (cc - expected) / np.sqrt(expected + 1.0)
    order = np.argsort(-surge, kind="stable")[:k]  # stable: equal surges keep ascending term id
    return ids[order].astype(np.int64), expected[order], surge[order]


def read_universe(path):
    """the tickers of a universe file: whitespace-separated entries, '#' starts a comment"""
    out = []
    with open(path, encoding="utf-8") as f:
        for line in f:
            out += line.split("#", 1)[0].split()
    return out


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m openintel_b200.trending",
                                 description="tickers ranked by the surge of their mentions against a baseline window (one GPU "
                                             "call for all terms)")
    ap.add_argument("--store", required=True, help="SQLite post store (openintel_b200.store schema)")
    ap.add_argument("--baseline-since", required=True, help="start of the baseline window, RFC 3339")
    ap.add_argument("--since", required=True, help="end of the baseline and start of the window, RFC 3339")
    ap.add_argument("--until", required=True, help="end of the window, RFC 3339")
    ap.add_argument("--top", type=int, default=20, help="how many terms to list (default 20)")
    ap.add_argument("--min-mentions", type=int, default=1, help="least mentions in the window to be ranked (default 1)")
    ap.add_argument("--source", choices=["reddit", "bluesky"], help="only this source's posts")
    ap.add_argument("--universe", help="file of tickers to rank among (whitespace-separated, '#' comments); default all")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args(argv)
    from . import capi, store, timeline
    try:
        t0, t1, t2 = (store.parse_created_at(x) for x in (args.baseline_since, args.since, args.until))
    except ValueError as e:
        ap.error(str(e))
    if not t0 < t1:
        ap.error("--baseline-since must be before --since")
    if not t1 < t2:
        ap.error("--since must be before --until")
    if args.top < 1:
        ap.error("--top must be at least 1")
    if args.min_mentions < 1:
        ap.error("--min-mentions must be at least 1")
    universe = None
    if args.universe is not None:
        try:
            universe = read_universe(args.universe)
        except (OSError, UnicodeDecodeError) as e:
            ap.error("--universe: %s" % e)
    conn = store.open_store(args.store)
    try:
        with store.MentionIndex(conn, device_index=args.device) as mi:
            ranked = mi.trending(t1, t2, t0, args.top, min_mentions=args.min_mentions, source=args.source, universe=universe)
    except (capi.OiError, ValueError) as e:  # a store without a token, a created_at without an offset
        sys.stderr.write("error: %s\n" % e)
        return 1
    finally:
        conn.close()
    out = {"baseline_since": timeline.format_time(t0), "since": timeline.format_time(t1), "until": timeline.format_time(t2),
           "source": args.source, "top": args.top, "min_mentions": args.min_mentions, "universe": args.universe,
           "ranked": ranked}
    sys.stdout.write(json.dumps(out) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
