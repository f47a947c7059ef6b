"""CPU side of the per-term timelines (SPEC §8b): the creation-time rule, the `--every` bucket edges and the time
window of analyze.select_posts."""
import pytest

from openintel_b200 import analyze, store, timeline


def test_parse_created_at_offsets_and_floor():
    P = store.parse_created_at
    assert P("1970-01-01T00:00:00Z") == 0
    assert P("2024-01-01T00:00:00Z") == 1704067200
    assert P("2024-01-01T00:00:00+00:00") == 1704067200
    assert P("2024-01-01T02:30:00+02:30") == 1704067200
    assert P("2023-12-31T19:00:00-05:00") == 1704067200
    # fractional seconds are floored, before and after the epoch
    assert P("2024-01-01T00:00:00.999999Z") == 1704067200
    assert P("2024-01-01T00:00:59.5+00:00") == 1704067259
    assert P("1969-12-31T23:59:59.5Z") == -1
    assert P("1969-12-31T23:59:59Z") == -1
    # so `t < E` is unchanged for every integer edge E
    assert P("2024-01-01T00:00:00.000001Z") < 1704067201
    for naive in ("2024-01-01T00:00:00", "2024-01-01 00:00:00", "2024-01-01"):
        with pytest.raises(ValueError):
            P(naive)
    with pytest.raises(ValueError):
        P("yesterday")


def test_every_and_bucket_edges():
    assert [timeline.parse_every(x) for x in ("1s", "90s", "5m", "1h", "24h", "1d", "7d")] == [1, 90, 300, 3600, 86400, 86400,
                                                                                             604800]
    for bad in ("0d", "d", "1w", "1.5h", "-1h", " 1h", "1hh", ""):
        with pytest.raises(ValueError):
            timeline.parse_every(bad)
    assert timeline.bucket_edges(0, 10, 3) == [0, 3, 6, 9, 10]
    assert timeline.bucket_edges(0, 9, 3) == [0, 3, 6, 9]
    assert timeline.bucket_edges(5, 6, 100) == [5, 6]
    jan = store.parse_created_at("2024-01-01T00:00:00Z")
    feb = store.parse_created_at("2024-02-01T00:00:00Z")
    e = timeline.bucket_edges(jan, feb, 86400)
    assert len(e) == 32 and e[0] == jan and e[-1] == feb and all(b - a == 86400 for a, b in zip(e, e[1:]))
    assert timeline.format_time(jan) == "2024-01-01T00:00:00Z" and timeline.format_time(e[1]) == "2024-01-02T00:00:00Z"
    assert timeline.format_time(-1) == "1969-12-31T23:59:59Z"
    for since, until in ((10, 10), (11, 10)):
        with pytest.raises(ValueError):
            timeline.bucket_edges(since, until, 1)


def _store(created):
    conn = store.open_store(":memory:")
    store.insert_posts(conn, [dict(id="p%d" % i, source=("reddit", "bluesky")[i % 2], author="a", text="post %d" % i,
                                   created_at=c, engagement=0) for i, c in enumerate(created)])
    return conn


def test_select_posts_window():
    # not in time order; p2 and p4 lie exactly on edges, p5 has a fraction and an offset
    created = ["2024-01-01T00:00:10Z", "2024-01-01T00:00:00Z", "2024-01-01T00:00:05Z", "2024-01-01T00:00:04.999Z",
               "2024-01-01T00:00:20Z", "2024-01-01T01:00:07.7+01:00"]
    conn = _store(created)
    t0 = store.parse_created_at("2024-01-01T00:00:00Z")
    ids = lambda **kw: analyze.select_posts(conn, **kw)[0]  # noqa: E731
    assert ids() == ["p%d" % i for i in range(6)]
    assert ids(since=t0 + 5, until=t0 + 20) == ["p0", "p2", "p5"]  # [since, until): p2 in, p4 out
    assert ids(since=t0 + 5) == ["p0", "p2", "p4", "p5"]
    assert ids(until=t0 + 5) == ["p1", "p3"]  # 4.999 s floors to 4
    assert ids(since=t0 + 7, until=t0 + 8) == ["p5"]
    assert ids(since=t0 + 21) == []
    # with source and limit: the window comes before the limit
    assert ids(source="reddit", since=t0 + 1) == ["p0", "p2", "p4"]
    assert ids(source="reddit", since=t0 + 1, limit=2) == ["p0", "p2"]
    assert ids(since=t0 + 10, limit=1) == ["p0"]
    conn.close()
    # a stored time without an offset is refused only when a window asks for the times, naming the post
    conn = _store(["2024-01-01T00:00:00Z", "2024-01-01T00:00:01"])
    assert ids() == ["p0", "p1"]
    with pytest.raises(ValueError) as e:
        ids(since=t0)
    assert "doc_id 1" in str(e.value)
    conn.close()


def test_social_block_is_the_report_social():
    sm = dict(total=3, bullish=2, bearish=0, neutral=1, net_sentiment=0.25, speculation_index=1 / 3, bull_bear_ratio=-1.0)
    block = analyze.social_block(sm, {"reddit": 2, "bluesky": 1})
    assert block == analyze.build_report(sm, {"reddit": 2, "bluesky": 1})["social"]
    assert list(block["mentions_by_source"]) == ["bluesky", "reddit"] and block["bull_bear_ratio"] is None
    assert analyze.social_block(analyze.empty_summary(), {"reddit": 0})["mentions_by_source"] == {}
