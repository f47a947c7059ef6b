"""The SPEC §8d ranking (related.rank) and the `related` CLI's argument checks: pure host code, no GPU."""
import math
import struct

import numpy as np
import pytest

from openintel_b200 import related

# anchor = term 0 with n_a = 10 posts of N = 100 in the window: expected = n_u / 10
CO = np.array([10, 8, 2, 0, 5, 1, 4, 3], dtype=np.uint32)
NU = np.array([10, 20, 20, 30, 10, 70, 40, 30], dtype=np.uint32)
#   expected:  -   2   2   3   1   7   4   3
#   score:     -  6/√3 0   -  4/√2 -6/√8 0  0     (term 3 has no co-mention)


def _bits(x):
    return struct.pack("<d", float(x))


def test_known_answer():
    ids, exp, score = related.rank(CO, NU, 10, 100, 0, k=100)
    # terms 2, 6 and 7 tie at 0: ascending term id; the anchor itself is never ranked
    assert ids.tolist() == [1, 4, 2, 6, 7, 5]
    assert exp.tolist() == [2.0, 1.0, 2.0, 4.0, 3.0, 7.0]
    assert score.tolist() == [(8 - 2) / math.sqrt(3), (5 - 1) / math.sqrt(2), 0.0, 0.0, 0.0, (1 - 7) / math.sqrt(8)]
    assert all(_bits(s) == _bits(0.0) for s in score[2:5])  # co == expected is +0.0


def test_min_co_mentions_k_and_anchor():
    assert related.rank(CO, NU, 10, 100, 0, k=100, min_co_mentions=3)[0].tolist() == [1, 4, 6, 7]
    assert related.rank(CO, NU, 10, 100, 0, k=2)[0].tolist() == [1, 4]
    assert related.rank(CO, NU, 10, 100, 0, k=5, min_co_mentions=11)[0].tolist() == []
    # no anchor left out: term 0 is ranked like any other term
    ids, _, score = related.rank(CO, NU, 10, 100, None, k=100)
    assert ids.tolist()[:3] == [0, 1, 4] and score[0] == (10 - 1) / math.sqrt(2)


def test_universe_mask():
    mask = np.zeros(len(CO), dtype=bool)
    mask[[0, 3, 5, 6]] = True  # term 0 is the anchor, term 3 has co = 0: neither is a candidate
    ids, exp, score = related.rank(CO, NU, 10, 100, 0, k=10, candidates=mask)
    assert ids.tolist() == [6, 5] and exp.tolist() == [4.0, 7.0]
    assert related.rank(CO, NU, 10, 100, 0, k=10, candidates=np.zeros(len(CO), dtype=bool))[0].tolist() == []


def test_n_edge_cases():
    # n_a = 0 (an anchor without a post in the window, N = 0 included) ranks nothing
    for n in (0, 100):
        ids, exp, score = related.rank(np.zeros(8, np.uint32), NU, 0, n, 0, k=10)
        assert ids.tolist() == [] and exp.tolist() == [] and score.tolist() == []
    # every post mentions the anchor (n_a = N): expected = n_u, so a term's score is (co - n_u) / sqrt(n_u + 1) = 0
    # when all its posts are the anchor's
    co = np.array([5, 3, 2], dtype=np.uint32)
    nu = np.array([5, 3, 2], dtype=np.uint32)
    ids, exp, score = related.rank(co, nu, 5, 5, 0, k=10)
    assert ids.tolist() == [1, 2] and exp.tolist() == [3.0, 2.0] and all(_bits(s) == _bits(0.0) for s in score)
    # one post in the window
    ids, exp, score = related.rank(np.array([1, 1], np.uint32), np.array([1, 1], np.uint32), 1, 1, 0, k=10)
    assert ids.tolist() == [1] and exp.tolist() == [1.0] and score.tolist() == [0.0]


def _rule(co, n_u, n_a, n_posts, anchor, k, min_co, allowed=None):
    """SPEC §8d in plain Python floats"""
    if n_a == 0:
        return []
    rows = []
    for u in range(len(co)):
        if u != anchor and int(co[u]) >= min_co and (allowed is None or u in allowed):
            e = (float(int(n_a)) * float(int(n_u[u]))) / float(int(n_posts))
            rows.append((u, e, (float(int(co[u])) - e) / math.sqrt(e + 1.0)))
    rows.sort(key=lambda r: (-r[2], r[0]))
    return rows[:k]


@pytest.mark.parametrize("n_posts", [400_000, 90_001, 3_999_999_999])
def test_expected_and_score_bit_for_bit_against_python_floats(n_posts):
    rng = np.random.default_rng(n_posts % 1000)
    n = 4000
    n_a = 70_000
    n_u = rng.integers(0, 90_000, n).astype(np.uint32)
    co = np.minimum(n_u, rng.integers(0, 3000, n)).astype(np.uint32)
    co[::13] = 0
    n_u[5::17] = n_u[4::17][:len(n_u[5::17])]  # equal n_u and co next to each other: ties
    co[5::17] = co[4::17][:len(co[5::17])]
    allowed = set(rng.choice(n, size=n // 3, replace=False).tolist())
    mask = np.zeros(n, dtype=bool)
    mask[list(allowed)] = True
    for k, mc, cand in ((n, 1, None), (50, 7, None), (n, 1, mask), (10, 3, mask)):
        ids, exp, score = related.rank(co, n_u, n_a, n_posts, 17, k, mc, cand)
        want = _rule(co, n_u, n_a, n_posts, 17, k, mc, None if cand is None else allowed)
        assert ids.tolist() == [u for u, _, _ in want]
        assert [_bits(x) for x in exp] == [_bits(e) for _, e, _ in want]
        assert [_bits(x) for x in score] == [_bits(s) for _, _, s in want]


def test_rank_refuses_bad_arguments():
    with pytest.raises(ValueError):
        related.rank(CO, NU[:-1], 10, 100, 0, 5)
    with pytest.raises(ValueError):
        related.rank(CO, NU, 10, 100, 0, 0)
    with pytest.raises(ValueError):
        related.rank(CO, NU, 10, 100, 0, 5, min_co_mentions=0)
    with pytest.raises(ValueError):
        related.rank(CO, NU, 10, 9, 0, 5)  # N < n_a
    for args in ((5, 5, 1, 1), (6, 5, 1, 1), (0, 1, 0, 1), (0, 1, 1, 0)):
        with pytest.raises(ValueError):
            related.check_args(*args)
    assert related.check_args(0, 1, 1, 1) == (0, 1, 1, 1)


def _usage_error(capsys, *argv):
    with pytest.raises(SystemExit) as e:
        related.main(list(argv))
    assert e.value.code == 2
    return capsys.readouterr().err


def test_cli_argument_errors(capsys, tmp_path):
    db = str(tmp_path / "never-opened.db")
    base = ["--store", db]
    t = ["2024-01-08T00:00:00Z", "2024-01-09T00:00:00Z"]
    err = _usage_error(capsys, *base, "--since", t[1], "--until", t[1], "GME")
    assert "--since must be before --until" in err
    err = _usage_error(capsys, *base, "--since", t[1], "--until", t[0], "GME")
    assert "--since must be before --until" in err
    err = _usage_error(capsys, *base, "--since", t[0], "--until", t[1], "--top", "0", "GME")
    assert "--top" in err
    err = _usage_error(capsys, *base, "--since", t[0], "--until", t[1], "--min-co-mentions", "0", "GME")
    assert "--min-co-mentions" in err
    err = _usage_error(capsys, *base, "--since", "yesterday", "--until", t[1], "GME")
    assert "yesterday" in err
    err = _usage_error(capsys, *base, "--since", "2024-01-08T00:00:00", "--until", t[1], "GME")
    assert "offset" in err
    err = _usage_error(capsys, *base, "--since", t[0], "--until", t[1], "--universe", str(tmp_path / "missing.txt"), "GME")
    assert "--universe" in err
    _usage_error(capsys, *base, "--since", t[0], "--until", t[1], "--source", "twitter", "GME")
    _usage_error(capsys, *base, "--since", t[0], "--until", t[1])  # no ticker
    _usage_error(capsys, "--since", t[0], "--until", t[1], "GME")  # --store is required
    assert not (tmp_path / "never-opened.db").exists()  # every refusal comes before the store is opened
