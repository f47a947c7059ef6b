"""The SPEC §8c ranking (trending.rank) and the `trending` CLI's argument checks: pure host code, no GPU."""
import math
import struct

import numpy as np
import pytest

from openintel_b200 import trending

# t0 = 0, t1 = 100, t2 = 150: the window is half the baseline, so expected = m / 2
C = np.array([5, 3, 10, 5, 0, 9, 1, 2], dtype=np.uint32)
M = np.array([0, 6, 30, 0, 8, 6, 0, 16], dtype=np.uint32)
#   surge:    5  0 -1.25 5  -   3  1  -2     (term 4 has no mention in the window)


def _bits(x):
    return struct.pack("<d", float(x))


def test_known_answer():
    ids, exp, surge = trending.rank(C, M, 0, 100, 150, k=100)
    # terms 0 and 3 tie at 5 (m = 0: surge = c): ascending term id
    assert ids.tolist() == [0, 3, 5, 6, 1, 2, 7]
    assert exp.tolist() == [0.0, 0.0, 3.0, 0.0, 3.0, 15.0, 8.0]
    assert surge.tolist() == [5.0, 5.0, 3.0, 1.0, 0.0, -1.25, -2.0]
    assert _bits(surge[4]) == _bits(0.0)  # c == expected is +0.0


def test_min_mentions_and_k():
    ids, _, surge = trending.rank(C, M, 0, 100, 150, k=100, min_mentions=2)
    assert ids.tolist() == [0, 3, 5, 1, 2, 7]  # term 6 (c = 1) is cut
    assert trending.rank(C, M, 0, 100, 150, k=3, min_mentions=2)[0].tolist() == [0, 3, 5]
    assert trending.rank(C, M, 0, 100, 150, k=1)[0].tolist() == [0]
    assert trending.rank(C, M, 0, 100, 150, k=5, min_mentions=11)[0].tolist() == []  # no candidate


def test_universe_mask():
    mask = np.zeros(len(C), dtype=bool)
    mask[[1, 3, 4, 7]] = True  # term 4 has c = 0: never a candidate
    ids, exp, surge = trending.rank(C, M, 0, 100, 150, k=10, candidates=mask)
    assert ids.tolist() == [3, 1, 7]  # k larger than the candidates: all of them
    assert exp.tolist() == [0.0, 3.0, 8.0] and surge.tolist() == [5.0, 0.0, -2.0]


def test_expected_and_surge_bit_for_bit_against_python_floats():
    rng = np.random.default_rng(8)
    n = 5000
    c = rng.integers(0, 4000, n).astype(np.uint32)
    m = rng.integers(0, 90000, n).astype(np.uint32)
    m[::7] = 0
    c[::11] = 0
    for t0, t1, t2 in ((1704067200, 1704067200 + 7 * 86400, 1704067200 + 8 * 86400), (-17, 4, 1_000_003), (0, 3, 10)):
        ids, exp, surge = trending.rank(c, m, t0, t1, t2, k=n)
        assert len(ids) == int(np.count_nonzero(c))
        want = {}
        for t in range(n):
            if c[t] >= 1:
                e = (float(int(m[t])) * float(t2 - t1)) / float(t1 - t0)
                want[t] = (e, (float(int(c[t])) - e) / math.sqrt(e + 1.0))
        for t, e, s in zip(ids.tolist(), exp, surge):
            assert _bits(e) == _bits(want[t][0]) and _bits(s) == _bits(want[t][1]), t
        # the order: surge descending, ties by ascending term id
        assert ids.tolist() == sorted(want, key=lambda t: (-want[t][1], t))


def test_rank_refuses_bad_arguments():
    for args in ((0, 0, 1, 5), (0, 2, 1, 5), (0, 1, 2, 0)):
        with pytest.raises(ValueError):
            trending.rank(C, M, *args)
    with pytest.raises(ValueError):
        trending.rank(C, M, 0, 1, 2, 5, min_mentions=0)
    with pytest.raises(ValueError):
        trending.rank(C, M[:-1], 0, 1, 2, 5)


def test_read_universe(tmp_path):
    p = tmp_path / "u.txt"
    p.write_text("$GME amc  # meme stocks\n\n# nothing here\nTSLA\n", encoding="utf-8")
    assert trending.read_universe(str(p)) == ["$GME", "amc", "TSLA"]


def _usage_error(capsys, *argv):
    with pytest.raises(SystemExit) as e:
        trending.main(list(argv))
    assert e.value.code == 2
    return capsys.readouterr().err


def test_cli_argument_errors(capsys, tmp_path):
    db = str(tmp_path / "never-opened.db")
    base = ["--store", db]
    t = ["2024-01-01T00:00:00Z", "2024-01-08T00:00:00Z", "2024-01-09T00:00:00Z"]
    err = _usage_error(capsys, *base, "--baseline-since", t[1], "--since", t[1], "--until", t[2])
    assert "--baseline-since must be before --since" in err
    err = _usage_error(capsys, *base, "--baseline-since", t[2], "--since", t[1], "--until", t[2])
    assert "--baseline-since must be before --since" in err
    err = _usage_error(capsys, *base, "--baseline-since", t[0], "--since", t[2], "--until", t[2])
    assert "--since must be before --until" in err
    err = _usage_error(capsys, *base, "--baseline-since", t[0], "--since", t[2], "--until", t[1])
    assert "--since must be before --until" in err
    err = _usage_error(capsys, *base, "--baseline-since", t[0], "--since", t[1], "--until", t[2], "--top", "0")
    assert "--top" in err
    err = _usage_error(capsys, *base, "--baseline-since", t[0], "--since", t[1], "--until", t[2], "--min-mentions", "0")
    assert "--min-mentions" in err
    err = _usage_error(capsys, *base, "--baseline-since", "yesterday", "--since", t[1], "--until", t[2])
    assert "yesterday" in err
    err = _usage_error(capsys, *base, "--baseline-since", "2024-01-01T00:00:00", "--since", t[1], "--until", t[2])
    assert "offset" in err
    err = _usage_error(capsys, *base, "--baseline-since", t[0], "--since", t[1], "--until", t[2], "--universe",
                       str(tmp_path / "missing.txt"))
    assert "--universe" in err
    _usage_error(capsys, *base, "--baseline-since", t[0], "--since", t[1], "--until", t[2], "--source", "twitter")
    _usage_error(capsys, "--since", t[1], "--until", t[2])  # --store and --baseline-since are required
    assert not (tmp_path / "never-opened.db").exists()  # every refusal comes before the store is opened
