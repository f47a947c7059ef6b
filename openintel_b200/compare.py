"""`python -m openintel_b200.compare` — the reference's `compare_tickers` (src/mcp/tools.rs:301-349) over a post store:
every ticker's `analyze --mention` report, ranked by one metric.

The reports come from store.MentionIndex: the posts that mention a ticker are its posting list in the index, so all
tickers are summarised in one device call instead of one pass over the store per ticker.  The ranking is the
reference's `sort_ranked` (tools.rs:283-299): descending by the metric, stable, so ties keep the order in which the
tickers were given.  A ticker with neither a mention nor a market snapshot, which `analyze` refuses with NoData, is
listed under "no_data" instead of failing the command.

    python -m openintel_b200.compare --store posts.db --by crowding --market GME=25.1,22.0,9000000,3000000 GME AMC BB
"""
import argparse
import json
import sys

from . import fusion

METRICS = {
    "speculation_index": lambda r: r["social"]["speculation_index"],
    "net_sentiment": lambda r: r["social"]["net_sentiment"],
    "total_mentions": lambda r: r["social"]["total_mentions"],
    "crowding": lambda r: r["fusion"]["crowding"],
}


def rank_reports(tickers, reports, by):
    """(ticker, report or None) pairs -> {"by", "ranked": [{"ticker", "value", "report"}], "no_data": [ticker]}"""
    metric = METRICS[by]
    ranked = [{"ticker": t, "value": metric(r), "report": r} for t, r in zip(tickers, reports) if r is not None]
    ranked.sort(key=lambda e: e["value"], reverse=True)  # stable: equal values keep the input order
    return {"by": by, "ranked": ranked, "no_data": [t for t, r in zip(tickers, reports) if r is None]}


def _market(ap, spec):
    """TICKER=last_price,previous_close,volume,avg_volume[,iv_rank] -> (ticker, fusion.MarketSummary)"""
    name, _, vals = spec.partition("=")
    f = vals.split(",")
    if not name or len(f) not in (4, 5):
        ap.error("--market takes TICKER=last_price,previous_close,volume,avg_volume[,iv_rank]")
    try:
        return name, fusion.MarketSummary.from_snapshot(float(f[0]), float(f[1]), int(f[2]), int(f[3]),
                                                        float(f[4]) if len(f) == 5 else None)
    except ValueError:
        ap.error("--market %s: not numbers" % spec)


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m openintel_b200.compare",
                                 description="rank tickers' speculation reports over stored posts (one GPU call for all)")
    ap.add_argument("--store", required=True, help="SQLite post store (openintel_b200.store schema)")
    ap.add_argument("--source", choices=["reddit", "bluesky"], help="only this source's posts")
    ap.add_argument("--by", choices=sorted(METRICS), default="speculation_index", help="ranking metric (descending)")
    ap.add_argument("--market", action="append", default=[], metavar="TICKER=last,prev,vol,avgvol[,iv]",
                    help="market snapshot of one ticker (repeatable)")
    ap.add_argument("--device", type=int, default=0)
    ap.add_argument("tickers", nargs="+", metavar="TICKER", help="cashtags / words, e.g. GME or $GME")
    args = ap.parse_args(argv)
    markets = dict(_market(ap, m) for m in args.market)
    from . import capi, store
    conn = store.open_store(args.store)
    try:
        with store.MentionIndex(conn, device_index=args.device) as mi:
            reports = mi.reports(args.tickers, source=args.source, markets=markets)
    except (capi.OiError, ValueError) as e:  # e.g. a store whose posts hold no token: nothing to index
        sys.stderr.write("error: %s\n" % e)
        return 1
    out = rank_reports(args.tickers, reports, args.by)
    out["source"] = args.source
    sys.stdout.write(json.dumps(out) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
