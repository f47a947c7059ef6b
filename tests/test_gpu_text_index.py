"""oi_index_build_bm25_text: the BM25 part built from post text on the device must equal, array for array, the CSR of the
host IndexBuilder on the same texts (SPEC §3 index layout), with the same vocabulary; the folded weights and the search
results of the two indexes are then bit-identical."""
import ctypes as C
import os

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu

DIM = 16


@pytest.fixture(scope="module")
def oi():
    import __graft_entry__ as ge  # noqa: F401
    import openintel_b200
    openintel_b200.load_library()
    import runpy
    from openintel_b200 import hostlib
    runpy.run_path(os.path.join(os.path.dirname(hostlib.__file__), "host", "build.py"), run_name="__build__")
    return openintel_b200


def _host(texts):
    from openintel_b200 import hostlib
    b = hostlib.IndexBuilder()
    b.add(texts)
    csr = b.finish()
    vocab = [b.term(i) for i in range(csr["n_terms"])]
    return b, csr, vocab


def _index(oi, n, max_batch=4):
    ix = oi.GpuIndex(n_docs=n, dim=DIM, max_k=10, max_batch=max_batch)
    from openintel_b200 import store
    ix.load_embeddings(store.normalise_rows_f32(O.synth_rows_f32(n, DIM) + np.float32(0.01)))
    return ix


def _check(oi, texts, queries=None):
    """device build == host builder: CSR, vocabulary, weights, BM25 and hybrid lists"""
    b, csr, vocab = _host(texts)
    n = len(texts)
    with _index(oi, n) as gx, _index(oi, n) as hx:
        got_vocab = gx.build_bm25_text(texts)
        assert gx.n_terms == csr["n_terms"]
        assert got_vocab == vocab
        gx.bm25_finalize()
        hx.load_bm25(csr["term_offsets"], csr["doc_ids"], csr["tfs"], csr["doc_len"])
        hx.bm25_finalize()
        P = len(csr["doc_ids"])
        g, h = gx.read_bm25(P), hx.read_bm25(P)
        for f in ("term_offsets", "doc_ids", "tfs", "doc_len"):
            assert np.array_equal(g[f], csr[f]), f
        assert np.array_equal(g["weights"].view(np.uint32), h["weights"].view(np.uint32))
        if queries is None:
            rng = np.random.default_rng(len(texts))
            queries = [rng.choice(csr["n_terms"], size=min(5, csr["n_terms"]), replace=False).astype(np.uint32) for _ in range(4)]
        qv = O.synth_rows_f32(len(queries), DIM, stream=1)
        qv /= np.linalg.norm(qv, axis=1, keepdims=True)
        for a, c in zip(gx.search_bm25(queries, 10), hx.search_bm25(queries, 10)):
            assert np.array_equal(a, c)
        for a, c in zip(gx.search_hybrid(qv, queries, 10), hx.search_hybrid(qv, queries, 10)):
            assert np.array_equal(a, c)
    b.close()
    return csr


def _zipf_posts(n_posts, n_words, seed):
    rng = np.random.default_rng(seed)
    alpha = np.frombuffer(b"abcdefghijklmnopqrstuvwxyz0123456789", dtype=np.uint8)
    lens = rng.integers(2, 15, size=n_words)
    chars = rng.choice(alpha, size=int(lens.sum()))
    cut = np.concatenate([[0], np.cumsum(lens)])
    words = [chars[cut[i]:cut[i + 1]].tobytes().decode() for i in range(n_words)]
    p = 1.0 / np.arange(1, n_words + 1)
    ntok = rng.integers(1, 40, size=n_posts)
    ids = rng.choice(n_words, size=int(ntok.sum()), p=p / p.sum())
    texts, at = [], 0
    for k in ntok:
        w = [words[i] for i in ids[at:at + k]]
        at += k
        texts.append(" ".join(x.capitalize() if j % 5 == 0 else x for j, x in enumerate(w)) + ("!" if k % 3 else ""))
    return texts


def test_configs0_corpus(oi):
    posts, _ = O.synth_posts(10000, 50000, O.SEED)
    csr = _check(oi, [p["text"] for p in posts])
    assert csr["n_terms"] > 1000


def test_200k_posts(oi):
    csr = _check(oi, _zipf_posts(200_000, 150_000, 7))
    assert len(csr["doc_ids"]) > 1_000_000


def test_adversarial_posts(oi):
    K = "\u212a"  # KELVIN SIGN: lowers to k
    base = "abcdefghijkl"  # 12 bytes
    texts = [
        K + "elvin mid" + K + "dle end" + K, "trunc \xe2\x84".encode("latin-1"), b"x\xe2\xe2\x84\xaay", "D\u0130ZZY \u0130stanbul s\u0130",
        "\u0130\u0130 a\u0130b " + K + K + " " + K,
        "MiXeD CaSe mixed CASE 0dte 0DTE a1b2C3 42 007 9", "",
        " ".join(base[:11] + base[:1] * j for j in range(0, 3)),
        " ".join([base, base + "a", base + "b", base + "0", base + "aa", base + "zzzz", base + "a" * 5, base + "z" * 88, base + "m" * 9988]),
        base + " " + base + "a " + base + " " + base + "a " + base + "b",
        "x" * 12 + " " + "x" * 13 + " " + "x" * 16 + " " + "x" * 17 + " " + "x" * 100 + " " + "x" * 10000 + " " + "x" * 11,
        ("lorem ipsum dolor " * 400) + base + "q" * 30,  # > 4096 bytes
        "!!! ??? ...", "\xff\xfe".encode("latin-1"), "solo",
        ("A" * 5000) + " tail",
        "\u00e9t\u00e9 caf\u00e9 na\u00efve \u00fcber",
    ]
    _check(oi, texts)
    _check(oi, ["only one post, with a few words: words"])
    # unaligned byte offsets: posts of every length 1..40 back to back
    _check(oi, ["ab" * (i // 2) + "c" * (i % 2) + " x%d" % i for i in range(1, 41)])


def test_random_bytes(oi):
    rng = np.random.default_rng(20261020)
    pool = np.frombuffer(b"aAzZ09 .,\xe2\x84\xaa\xc4\xb0\xff\x80", dtype=np.uint8)
    texts = []
    for i in range(3000):
        n = int(rng.integers(0, 300))
        if i % 3 == 0:
            texts.append(rng.integers(0, 256, size=n, dtype=np.uint8).tobytes())  # any bytes, invalid UTF-8 included
        else:
            texts.append(rng.choice(pool, size=n).tobytes())
    _check(oi, texts)


def _raw_build(ix, blob, offs, n):
    nt, nb = C.c_uint32(), C.c_uint64()
    return ix.L.oi_index_build_bm25_text(ix.h, blob, offs, n, C.byref(nt), C.byref(nb))


def test_errors_leave_no_bm25_part(oi):
    texts = ["alpha beta", "beta gamma", "gamma"]
    from openintel_b200 import capi
    blob, offs = capi.pack_texts(texts)
    q = [np.array([0], dtype=np.uint32)]
    with _index(oi, 3) as ix:
        launches = ix.launch_count()
        ix.build_bm25_text(texts)
        assert ix.launch_count() > launches
        ix.bm25_finalize()
        ix.search_bm25(q, 3)
        # n_posts != n_docs
        assert _raw_build(ix, blob.ctypes.data, offs.ctypes.data, 2) == 1
        with pytest.raises(oi.OiError) as e:
            ix.search_bm25(q, 3)
        assert e.value.status == 5
        # decreasing offsets, NULL pointers
        bad = offs.copy()
        bad[2] = 1
        assert _raw_build(ix, blob.ctypes.data, bad.ctypes.data, 3) == 1
        assert _raw_build(ix, None, offs.ctypes.data, 3) == 1
        assert _raw_build(ix, blob.ctypes.data, None, 3) == 1
        assert ix.L.oi_index_build_bm25_text(ix.h, blob.ctypes.data, offs.ctypes.data, 3, None, None) == 1
        # a good build after failures works again
        ix.build_bm25_text(texts)
        ix.bm25_finalize()
        ix.search_bm25(q, 3)
        # a corpus without any token
        with pytest.raises(oi.OiError) as e:
            ix.build_bm25_text(["!!!", "", "\xff".encode("latin-1")])
        assert e.value.status == 1 and "no token" in e.value.message
        with pytest.raises(oi.OiError) as e:
            ix.search_bm25(q, 3)
        assert e.value.status == 5
        vo = np.empty(4, dtype=np.uint64)
        vb = np.empty(64, dtype=np.uint8)
        assert ix.L.oi_index_read_vocabulary(ix.h, vb.ctypes.data, vo.ctypes.data) == 5


def test_build_replaces_a_loaded_csr_and_the_other_way(oi):
    first, second = ["one two three", "two three", "three"], ["four five", "five six seven", "seven"]
    _, c1, _ = _host(first)
    _, c2, v2 = _host(second)
    vo = np.empty(16, dtype=np.uint64)
    vb = np.empty(64, dtype=np.uint8)
    with _index(oi, 3) as ix:
        ix.load_bm25(c1["term_offsets"], c1["doc_ids"], c1["tfs"], c1["doc_len"])
        assert ix.L.oi_index_read_vocabulary(ix.h, vb.ctypes.data, vo.ctypes.data) == 5  # a CSR-loaded index has none
        assert ix.build_bm25_text(second) == v2
        ix.bm25_finalize()
        g = ix.read_bm25(len(c2["doc_ids"]))
        for f in ("term_offsets", "doc_ids", "tfs", "doc_len"):
            assert np.array_equal(g[f], c2[f]), f
        assert ix.L.oi_index_read_vocabulary(ix.h, vb.ctypes.data, vo.ctypes.data) == 0
        ix.load_bm25(c1["term_offsets"], c1["doc_ids"], c1["tfs"], c1["doc_len"])  # drops the vocabulary
        assert ix.L.oi_index_read_vocabulary(ix.h, vb.ctypes.data, vo.ctypes.data) == 5


def test_store_index_query_terms_match_the_host_builder(oi, tmp_path):
    from openintel_b200 import store
    n, vocab, dim = 3000, 800, 32
    posts, _ = O.synth_posts(n, vocab, O.SEED)
    conn = store.open_store(str(tmp_path / "posts.db"), dim=dim)
    store.insert_posts(conn, posts, O.synth_rows_f32(n, dim))
    texts = ["%s %s, $%s zzzunknown %s" % tuple(posts[37]["text"].split()[:3] + [posts[37]["text"].split()[0]]),
             " ".join(posts[n // 2]["text"].split()[:8]), "nothingmatches here", "W1 w1 W2 w%d" % (vocab - 1), ""]
    b, csr, _ = store.lift_csr(conn)
    with store.StoreIndex(conn, max_k=10, max_batch=8) as sx:
        assert sx.n_terms == csr["n_terms"]
        assert [sx.builder.term(i) for i in range(sx.n_terms)] == [b.term(i) for i in range(csr["n_terms"])]
        got = sx.query_terms(texts)
        for j, t in enumerate(texts):
            assert got[j].tolist() == list(dict.fromkeys(b.query_terms(t).tolist()))
            assert sx.builder.query_terms(t).tolist() == b.query_terms(t).tolist()
        g = sx.ix.read_bm25(len(csr["doc_ids"]))
        for f in ("term_offsets", "doc_ids", "tfs", "doc_len"):
            assert np.array_equal(g[f], csr[f]), f
    b.close()
    conn.close()
