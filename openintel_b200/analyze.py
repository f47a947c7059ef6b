"""`python -m openintel_b200.analyze` — the reference's `analyze` use case (src/application/analyze.rs:16-73) over the posts
of a SQLite post store, with the GPU PostAnalyzer in the seat of `LexiconAnalyzer`:

    posts (store) -> GpuLexicon: per-post (polarity, speculative) + the social summary, one device call
                  -> fusion signals on the host (fusion.py: crowding, alignment, confidence)
                  -> a report shaped like the reference's SpeculationReport (src/domain/entities/speculation_report.rs)

The reference fetches a ticker's posts from its HTTP sources; here they are already stored, so the request selects them
(all, one source, or those that mention a cashtag / word).  An optional market snapshot (last price, previous close,
volume, average volume, IV rank) feeds the fusion exactly as `SpeculationEngine::aggregate` does.  No CPU analyzer path.
"""
import argparse
import json
import sys
from collections import OrderedDict

from . import capi, fusion

DISCLAIMER = "Informational only; not investment advice."


class NoData(ValueError):
    """DomainError::NoData (src/application/analyze.rs:58-60): neither posts nor a market snapshot"""


def ticker_key(text):
    """a ticker or mention word as the index holds it: the leading '$' dropped (the reference's tokenizer drops it
    too), lower case"""
    return text.lstrip("$").lower()


def select_posts(conn, source=None, mention=None, limit=None, since=None, until=None):
    """(ids, sources, texts) of the stored posts in doc order; `mention`: keep posts one of whose tokens equals it
    (normalised by ticker_key); `since` / `until`: keep posts
    created in [since, until), seconds since the Unix epoch (store.parse_created_at; SPEC §8b), before `limit`"""
    window = since is not None or until is not None
    sql, args = "SELECT id, source, text%s FROM posts" % (", doc_id, created_at" if window else ""), []
    if source:
        sql += " WHERE source = ?"
        args.append(source)
    sql += " ORDER BY doc_id"
    rows = conn.execute(sql, args).fetchall()
    if window:
        from .store import parse_created_at
        kept = []
        for r in rows:
            try:
                t = parse_created_at(r[4])
            except ValueError as e:
                raise ValueError("post doc_id %d: %s" % (r[3], e)) from None
            if (since is None or t >= since) and (until is None or t < until):
                kept.append(r)
        rows = kept
    if mention:
        from . import hostlib
        want = ticker_key(mention)
        rows = [r for r in rows if want in hostlib.tokenize(r[2])]
    if limit is not None:
        rows = rows[:limit]
    return [r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows]


def empty_summary():
    """the social summary of no posts (SpeculationEngine::social_summary over an empty slice; -1 = no bearish post)"""
    return dict(total=0, bullish=0, bearish=0, neutral=0, net_sentiment=0.0, speculation_index=0.0, bull_bear_ratio=-1.0)


def social_block(sm, mentions_by_source):
    """the "social" block of a report (the reference's SocialSummary as SpeculationReport shows it): sm: a summary dict
    shaped like GpuLexicon's; mentions_by_source: {source name: post count}"""
    by_source = OrderedDict()
    for s in sorted(mentions_by_source):  # the reference keeps a BTreeMap: sorted keys
        if mentions_by_source[s]:
            by_source[s] = int(mentions_by_source[s])
    return {"total_mentions": int(sm["total"]), "mentions_by_source": by_source, "net_sentiment": sm["net_sentiment"],
            "bullish": int(sm["bullish"]), "bearish": int(sm["bearish"]), "neutral": int(sm["neutral"]),
            "bull_bear_ratio": None if sm["bull_bear_ratio"] < 0 else sm["bull_bear_ratio"],
            "speculation_index": sm["speculation_index"]}


def build_report(sm, mentions_by_source, market=None, cfg=fusion.EngineConfig()):
    """The rest of SpeculationEngine::aggregate (src/domain/engine/speculation_engine.rs:21-66) once the social summary
    is known: the fusion signals and a report shaped like the reference's SpeculationReport.  sm: a summary dict shaped
    like GpuLexicon's; mentions_by_source: {source name: post count}; market: fusion.MarketSummary or None.  Raises
    NoData when there is neither a post nor a market snapshot."""
    if sm["total"] == 0 and market is None:
        raise NoData("no posts and no market snapshot")
    notes = []
    if market is None:
        notes.append("social-only, no price reference")
    social = social_block(sm, mentions_by_source)

    class _S:
        total, net_sentiment, speculation_index = social["total_mentions"], social["net_sentiment"], social["speculation_index"]
    fz = fusion.fuse(_S, market, cfg)
    return {"social": social,
            "market": None if market is None else {"pct_change": market.pct_change, "rvol": market.rvol, "iv_rank": market.iv_rank},
            "fusion": {"alignment": fz["alignment"], "crowding": fz["crowding"], "notes": notes},
            "social_confidence": fz["social_confidence"], "disclaimer": DISCLAIMER}


def analyze_posts(lexicon, sources, texts, market=None, cfg=fusion.EngineConfig()):
    """SpeculationEngine::aggregate (src/domain/engine/speculation_engine.rs:21-66) with the signals and the social
    summary coming from ONE GPU call.  market: fusion.MarketSummary or None."""
    if len(sources) != len(texts):
        raise ValueError("analyzer mismatch: %d sources for %d posts" % (len(sources), len(texts)))
    if texts:
        pol, spec, _, _, sm = lexicon.analyze(texts, summary=True, threshold=cfg.bull_bear_threshold)
    else:
        pol, spec, sm = [], [], empty_summary()
    report = build_report(sm, {s: sources.count(s) for s in set(sources)}, market, cfg)
    return report, pol, spec


def main(argv=None):
    ap = argparse.ArgumentParser(prog="python -m openintel_b200.analyze", description="speculation report over stored posts (GPU PostAnalyzer)")
    ap.add_argument("--store", required=True, help="SQLite post store (openintel_b200.store schema)")
    ap.add_argument("--source", choices=["reddit", "bluesky"], help="only this source's posts")
    ap.add_argument("--mention", help="only posts that mention this cashtag / word (e.g. GME)")
    ap.add_argument("--since", help="only posts created at or after this RFC 3339 time (e.g. 2024-01-01T00:00:00Z)")
    ap.add_argument("--until", help="only posts created before this RFC 3339 time")
    ap.add_argument("--limit", type=int, help="at most this many posts")
    ap.add_argument("--market", help="last_price,previous_close,volume,avg_volume[,iv_rank]")
    ap.add_argument("--device", type=int, default=0)
    args = ap.parse_args(argv)
    from . import store
    market = None
    if args.market:
        f = args.market.split(",")
        if len(f) not in (4, 5):
            ap.error("--market takes last_price,previous_close,volume,avg_volume[,iv_rank]")
        market = fusion.MarketSummary.from_snapshot(float(f[0]), float(f[1]), int(f[2]), int(f[3]), float(f[4]) if len(f) == 5 else None)
    since = until = None
    try:
        if args.since is not None:
            since = store.parse_created_at(args.since)
        if args.until is not None:
            until = store.parse_created_at(args.until)
    except ValueError as e:
        ap.error("--since / --until: %s" % e)
    conn = store.open_store(args.store)
    try:
        _, sources, texts = select_posts(conn, args.source, args.mention, args.limit, since, until)
    except ValueError as e:  # a stored created_at that is not RFC 3339 with an offset
        sys.stderr.write("error: %s\n" % e)
        return 1
    with capi.GpuLexicon(args.device) as lx:
        try:
            report, _, _ = analyze_posts(lx, sources, texts, market)
        except NoData as e:
            sys.stderr.write("error: %s\n" % e)
            return 1
    sys.stdout.write(json.dumps(report) + "\n")
    return 0


if __name__ == "__main__":
    sys.exit(main())
