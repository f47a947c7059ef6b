"""The SPEC §8e figures, order and merge (authors.rank, authors.merge) and the `authors` CLI's argument checks: pure host
code, no GPU."""
import struct

import numpy as np
import pytest

from openintel_b200 import authors, capi


def _bits(x):
    return struct.pack("<d", float(x))


def _runs(rows, term=0):
    """[(author, posts, engagement)] -> AUTHOR_RUN_DTYPE runs of one term"""
    out = np.zeros(len(rows), dtype=capi.AUTHOR_RUN_DTYPE)
    for i, (a, p, e) in enumerate(rows):
        out[i]["term"], out[i]["author"], out[i]["posts"], out[i]["engagement"] = term, a, p, e
        out[i]["bullish"], out[i]["bearish"], out[i]["speculative"] = p // 2, p // 4, p // 3
        out[i]["first_at"], out[i]["last_at"] = 1000 + a, 2000 + a * p
    return out


def test_known_answer():
    # P = 10, S = 36 + 9 + 1 = 46: hhi = 46 / 100, effective_authors = 100 / 46; k = 2: top_share = 9 / 10
    r = authors.rank(_runs([(4, 3, 0), (7, 6, 5), (2, 1, 9)]), 2)
    assert r["mentions"] == 10 and r["authors"] == 3 and r["engagement"] == 14
    assert _bits(r["hhi"]) == _bits(46 / 100) and _bits(r["effective_authors"]) == _bits(100 / 46)
    assert _bits(r["top_share"]) == _bits(9 / 10)
    assert r["top"]["author"].tolist() == [7, 4] and r["top"]["posts"].tolist() == [6, 3]
    # one author: all the talk is theirs
    r = authors.rank(_runs([(3, 500, 12)]), 10)
    assert (r["hhi"], r["effective_authors"], r["top_share"]) == (1.0, 1.0, 1.0) and r["top"]["author"].tolist() == [3]
    # 500 authors with one post each
    r = authors.rank(_runs([(a, 1, 0) for a in range(500)]), 10)
    assert r["effective_authors"] == 500.0 and r["hhi"] == 1 / 500 and r["top_share"] == 10 / 500
    assert r["top"]["author"].tolist() == list(range(10))  # all tied: ascending author id


def test_order_and_its_ties():
    # equal posts -> engagement descending; equal posts and engagement -> author ascending
    rows = [(9, 5, 1), (1, 5, 1), (5, 5, 7), (3, 2, 100), (0, 5, 1), (8, 7, 0), (2, 2, 100), (6, 2, 2 ** 40)]
    r = authors.rank(_runs(rows), 100)
    assert r["top"]["author"].tolist() == [8, 5, 0, 1, 9, 6, 2, 3]
    assert authors.rank(_runs(rows), 3)["top"]["author"].tolist() == [8, 5, 0]
    # the input order does not matter
    perm = np.random.default_rng(3).permutation(len(rows))
    assert authors.rank(_runs(rows)[perm], 100)["top"].tobytes() == r["top"].tobytes()


def test_no_post():
    for runs in (_runs([]), _runs([(1, 0, 0), (2, 0, 0)])):
        r = authors.rank(runs, 5)
        assert r["mentions"] == 0 and r["hhi"] == 0.0 and r["effective_authors"] == 0.0 and r["top_share"] == 0.0
        assert len(r["top"]) == 0
    assert authors.rank(_runs([]), 5)["authors"] == 0


def _rule(rows, k):
    """SPEC §8e in plain Python ints and floats: (hhi, effective_authors, top_share, ranked authors)"""
    P = sum(p for _, p, _ in rows)
    S = sum(p * p for _, p, _ in rows)
    ranked = sorted(rows, key=lambda r: (-r[1], -r[2], r[0]))[:k]
    return (float(S) / (float(P) * float(P)), (float(P) * float(P)) / float(S),
            float(sum(p for _, p, _ in ranked)) / float(P), [a for a, _, _ in ranked])


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_figures_bit_for_bit_against_python_floats(seed):
    rng = np.random.default_rng(seed)
    n = 3000
    posts = rng.zipf(1.6, n).clip(1, 2 ** 20)  # large P and S: f64 rounding of S and P*P is exercised
    posts[:5] = 2 ** 26 + rng.integers(0, 1000, 5)
    eng = rng.integers(0, 4, n) * (2 ** 33)
    rows = [(int(a), int(p), int(e)) for a, p, e in zip(rng.permutation(n) * 3, posts, eng)]
    for k in (1, 10, n):
        r = authors.rank(_runs(rows), k)
        hhi, eff, share, ranked = _rule(rows, k)
        assert _bits(r["hhi"]) == _bits(hhi) and _bits(r["effective_authors"]) == _bits(eff)
        assert _bits(r["top_share"]) == _bits(share)
        assert r["top"]["author"].tolist() == ranked
        assert r["mentions"] == sum(p for _, p, _ in rows) and r["authors"] == n


def test_merge_of_a_run_split_over_three_ranks():
    whole = _runs([(4, 9, 30), (7, 2, 1)], term=1)
    whole[0]["first_at"], whole[0]["last_at"] = 100, 900
    parts = []
    for posts, bull, bear, spec, eng, lo, hi in ((3, 2, 1, 0, 10, 400, 500), (5, 1, 1, 2, 20, 100, 900),
                                                 (1, 1, 0, 1, 0, 300, 300)):
        p = _runs([(4, posts, eng)], term=1)
        p["bullish"], p["bearish"], p["speculative"], p["first_at"], p["last_at"] = bull, bear, spec, lo, hi
        parts.append(p)
    whole[0]["bullish"], whole[0]["bearish"], whole[0]["speculative"] = 4, 2, 3
    other = _runs([(7, 2, 1)], term=1)
    term0 = _runs([(4, 1, 1)], term=0)
    got = authors.merge([np.concatenate([parts[2], other]), parts[0], np.concatenate([parts[1], term0])])
    assert got.tobytes() == np.concatenate([term0, whole]).tobytes()
    # any order of the ranks gives the same runs
    assert authors.merge([parts[1], term0, other, parts[0], parts[2]]).tobytes() == got.tobytes()
    assert authors.merge([]).size == 0 and authors.merge([_runs([])]).size == 0
    assert authors.merge([whole]).tobytes() == whole.tobytes()


def test_rank_and_check_args_refuse_bad_arguments():
    with pytest.raises(ValueError):
        authors.rank(_runs([(1, 1, 1)]), 0)
    for args in ((5, 5, 1), (6, 5, 1), (0, 1, 0)):
        with pytest.raises(ValueError):
            authors.check_args(*args)
    assert authors.check_args(0, 1, 1) == (0, 1, 1)


def _usage_error(capsys, *argv):
    with pytest.raises(SystemExit) as e:
        authors.main(list(argv))
    assert e.value.code == 2
    return capsys.readouterr().err


def test_cli_argument_errors(capsys, tmp_path):
    db = str(tmp_path / "never-opened.db")
    base = ["--store", db]
    t = ["2024-01-08T00:00:00Z", "2024-01-09T00:00:00Z"]
    assert "--since must be before --until" in _usage_error(capsys, *base, "--since", t[1], "--until", t[1], "GME")
    assert "--since must be before --until" in _usage_error(capsys, *base, "--since", t[1], "--until", t[0], "GME")
    assert "--top" in _usage_error(capsys, *base, "--since", t[0], "--until", t[1], "--top", "0", "GME")
    assert "yesterday" in _usage_error(capsys, *base, "--since", "yesterday", "--until", t[1], "GME")
    assert "offset" in _usage_error(capsys, *base, "--since", "2024-01-08T00:00:00", "--until", t[1], "GME")
    _usage_error(capsys, *base, "--since", t[0], "--until", t[1], "--source", "twitter", "GME")
    _usage_error(capsys, *base, "--since", t[0], "--until", t[1])  # no ticker
    _usage_error(capsys, "--since", t[0], "--until", t[1], "GME")  # --store is required
    assert not (tmp_path / "never-opened.db").exists()  # every refusal comes before the store is opened
