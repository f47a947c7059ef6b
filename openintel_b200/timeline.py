"""`python -m openintel_b200.timeline` — how the social summary of tickers moved over time, over a post store: per
ticker, the "social" block of `analyze --mention T --since a --until b` for every time bucket [a, b) (SPEC §8b).

The blocks come from store.MentionIndex.timeline: a bucket splits a ticker's posting list into doc-order pieces, so all
tickers and all buckets are summarised in one device call instead of one pass over the store per ticker and bucket.
The buckets are `since + i * every`; the last one ends at `until` (and is shorter when `every` does not divide the
span).

    python -m openintel_b200.timeline --store posts.db --since 2024-01-01T00:00:00Z --until 2024-02-01T00:00:00Z \\
        --every 1d [--source reddit] GME AMC
"""
import argparse
import datetime
import json
import re
import sys

UNITS = {"s": 1, "m": 60, "h": 3600, "d": 86400}


def parse_every(text):
    """'Ns' | 'Nm' | 'Nh' | 'Nd' (N a positive integer) -> seconds"""
    m = re.fullmatch(r"([0-9]+)([smhd])", text)
    if not m or int(m.group(1)) == 0:
        raise ValueError("--every takes Ns, Nm, Nh or Nd with N > 0, not %r" % (text,))
    return int(m.group(1)) * UNITS[m.group(2)]


def bucket_edges(since, until, every):
    """[since, since + every, since + 2 every, ..., until]: the buckets [edges[b], edges[b + 1]), the last one ending at
    until"""
    if not since < until:
        raise ValueError("--since must be before --until")
    return list(range(since, until, every)) + [until]


def format_time(seconds):
    """seconds since the Unix epoch -> YYYY-MM-DDTHH:MM:SSZ"""
    return (datetime.datetime(1970, 1, 1) + datetime.timedelta(seconds=seconds)).strftime("%Y-%m-%dT%H:%M:%SZ")


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m openintel_b200.timeline",
                                 description="tickers' social summaries per time bucket over stored posts (one GPU call)")
    ap.add_argument("--store", required=True, help="SQLite post store (openintel_b200.store schema)")
    ap.add_argument("--since", required=True, help="start of the first bucket, RFC 3339 (e.g. 2024-01-01T00:00:00Z)")
    ap.add_argument("--until", required=True, help="end of the last bucket, RFC 3339")
    ap.add_argument("--every", required=True, help="bucket width: Ns, Nm, Nh or Nd")
    ap.add_argument("--source", choices=["reddit", "bluesky"], help="only this source's posts")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("tickers", nargs="+", metavar="TICKER", help="cashtags / words, e.g. GME or $GME")
    args = ap.parse_args(argv)
    from . import capi, store
    try:
        edges = bucket_edges(store.parse_created_at(args.since), store.parse_created_at(args.until), parse_every(args.every))
    except ValueError as e:
        ap.error(str(e))
    conn = store.open_store(args.store)
    try:
        with store.MentionIndex(conn, device_index=args.device) as mi:
            blocks = mi.timeline(args.tickers, edges, source=args.source)
    except (capi.OiError, ValueError) as e:  # a store without a token, a created_at without an offset
        sys.stderr.write("error: %s\n" % e)
        return 1
    finally:
        conn.close()
    out = {"source": args.source, "every": args.every,
           "buckets": [[format_time(a), format_time(b)] for a, b in zip(edges, edges[1:])],
           "tickers": [{"ticker": t, "timeline": b} for t, b in zip(args.tickers, blocks)]}
    sys.stdout.write(json.dumps(out) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
