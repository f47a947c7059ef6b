"""oi_index_bm25_union_vocabulary and the device lift of a document-sharded index (SPEC §5): every shard builds its doc
range from text on the device, the shards' vocabularies are united and each shard's lists are re-indexed to the global
term ids.  The shards must add up to the unsharded build array for array, rank like it bit for bit, and equal the host
lift (store.lift_shard) of the same rank."""
import ctypes as C
import os
import socket

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu

DIM, K = 16, 10


@pytest.fixture(scope="module")
def oi():
    import __graft_entry__ as ge  # noqa: F401
    import openintel_b200
    openintel_b200.load_library()
    import runpy
    from openintel_b200 import hostlib
    runpy.run_path(os.path.join(os.path.dirname(hostlib.__file__), "host", "build.py"), run_name="__build__")
    return openintel_b200


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


def _adversarial_posts():
    """24 posts: with 8 shards of 3 (or 3 of 8, 2 of 12) the tokens sharing a 12-byte prefix, the U+0130 / KELVIN SIGN
    tokens and the terms of one shard only land in different shards, and every shard holds a token"""
    Kv = "\u212a"  # KELVIN SIGN: lowers to k
    base = "abcdefghijkl"  # 12 bytes
    return [
        base + " " + base + "a onlyshardzero",
        Kv + "elvin mid" + Kv + "dle end" + Kv,
        "!!! ??? ...",
        base + "b " + base + "0 " + base + "aa",
        "D\u0130ZZY \u0130stanbul s\u0130",
        "",
        base + "zzzz " + base + "a" * 5 + " onlyshardtwo",
        "\u0130\u0130 a\u0130b " + Kv + Kv + " " + Kv,
        "trunc \xe2\x84".encode("latin-1"),
        base + "z" * 88 + " " + base + "m" * 9988,
        "MiXeD CaSe mixed CASE 0dte 0DTE a1b2C3 42 007 9",
        "x" * 12 + " " + "x" * 13 + " " + "x" * 16 + " " + "x" * 100 + " " + "x" * 10000 + " " + "x" * 11,
        " ".join(base[:11] + base[:1] * j for j in range(0, 3)),
        b"x\xe2\xe2\x84\xaay",
        ("lorem ipsum dolor " * 400) + base + "q" * 30,
        "\xff\xfe".encode("latin-1"),
        "solo",
        ("A" * 5000) + " tail",
        "\u00e9t\u00e9 caf\u00e9 na\u00efve \u00fcber",
        base + " " + base + "a " + base + " " + base + "m" * 9988,
        Kv + "elvin " + base + "zzzz",
        "\u0130stanbul kelvin " + "x" * 13,
        "xxxxxxxxxxxxy " + "x" * 10000,
        "lastshardonly word",
    ]


@pytest.fixture(scope="module")
def corpora():
    posts, _ = O.synth_posts(10000, 50000, O.SEED)
    return {"configs0": [p["text"] for p in posts], "zipf200k": _zipf_posts(200_000, 150_000, 7),
            "adversarial": _adversarial_posts()}


def _host(texts):
    from openintel_b200 import hostlib
    b = hostlib.IndexBuilder()
    b.add(texts)
    csr = b.finish()
    vocab = [b.term(i) for i in range(csr["n_terms"])]
    b.close()
    return csr, vocab


def _rows(n):
    from openintel_b200 import store
    return store.normalise_rows_f32(O.synth_rows_f32(n, DIM) + np.float32(0.01))


def _read_csr(ix, n_postings):
    """the BM25 part's CSR (no weights: readable before finalize)"""
    to = np.empty(ix.n_terms + 1, dtype=np.uint64)
    di = np.empty(max(n_postings, 1), dtype=np.uint32)
    tf = np.empty(max(n_postings, 1), dtype=np.uint32)
    dl = np.empty(ix.n_docs, dtype=np.uint32)
    ix._ck(ix.L.oi_index_read_bm25(ix.h, to.ctypes.data, di.ctypes.data, tf.ctypes.data, dl.ctypes.data, None))
    return dict(term_offsets=to, doc_ids=di[:n_postings], tfs=tf[:n_postings], doc_len=dl)


def _shards(oi, texts, world, rows):
    """one GpuIndex per shard on this GPU, each built from its slice and united with the gathered vocabularies"""
    from openintel_b200 import sharding
    shards = []
    for r in range(world):
        base, n = sharding.shard_range(len(texts), world, r)
        ix = oi.GpuIndex(n_docs=n, dim=DIM, doc_base=base, max_k=K, max_batch=4)
        ix.load_embeddings(rows[base:base + n])
        ix.build_bm25_text(texts[base:base + n])
        shards.append(ix)
    packed = [ix.read_vocabulary_packed() for ix in shards]
    blob = np.concatenate([b for b, _ in packed])
    offs = np.concatenate([[0], np.cumsum(np.concatenate([np.diff(o.astype(np.int64)) for _, o in packed]))]).astype(np.uint64)
    vocabs = [ix.bm25_union_vocabulary(blob, offs) for ix in shards]
    return shards, vocabs


def _check_shards(shards, vocabs, csr, vocab):
    """every shard has the global vocabulary; the shards' lists concatenate to the unsharded ones"""
    G, P = csr["n_terms"], len(csr["doc_ids"])
    terms, docs, tfs, dls = [], [], [], []
    df = np.zeros(G, dtype=np.uint64)
    total_off = np.zeros(G + 1, dtype=np.uint64)
    for ix, v in zip(shards, vocabs):
        assert v == vocab and ix.n_terms == G
        b, o = ix.read_vocabulary_packed()
        assert [bytes(b[o[t]:o[t + 1]]).decode() for t in range(G)] == vocab
        ldf, _, npost = ix.bm25_local_stats()
        c = _read_csr(ix, npost)
        assert c["term_offsets"][0] == 0 and c["term_offsets"][-1] == npost
        lens = np.diff(c["term_offsets"])
        assert np.array_equal(ldf, lens.astype(np.uint32))
        df += lens
        total_off += c["term_offsets"]
        terms.append(np.repeat(np.arange(G), lens.astype(np.int64)))
        docs.append(c["doc_ids"].astype(np.int64) + ix.doc_base)
        tfs.append(c["tfs"])
        dls.append(c["doc_len"])
    order = np.argsort(np.concatenate(terms), kind="stable")  # shards in doc order: each term's lists concatenate
    assert np.array_equal(total_off, csr["term_offsets"])
    assert np.array_equal(np.concatenate(docs)[order], csr["doc_ids"].astype(np.int64))
    assert np.array_equal(np.concatenate(tfs)[order], csr["tfs"])
    assert np.array_equal(np.concatenate(dls), csr["doc_len"])
    assert np.array_equal(df, np.diff(csr["term_offsets"]))
    assert P == int(df.sum())


def _finalize_global(shards, n_docs):
    dfs, sdl = [], 0
    for ix in shards:
        df, s, _ = ix.bm25_local_stats()
        dfs.append(df.astype(np.uint64))
        sdl += s
    gdf = np.sum(dfs, axis=0).astype(np.uint32)
    avgdl = float(np.float32(np.float64(sdl) / n_docs))
    for ix in shards:
        ix.bm25_finalize(avgdl=avgdl, n_docs_global=n_docs, global_df=gdf)


def _queries(csr, vocab, seed):
    rng = np.random.default_rng(seed)
    G = csr["n_terms"]
    df = np.diff(csr["term_offsets"])
    rare = np.flatnonzero(df == 1)  # terms of one post, hence of one shard
    q = [rng.choice(G, size=min(5, G), replace=False).astype(np.uint32),
         rng.choice(G, size=min(3, G), replace=False).astype(np.uint32),
         np.concatenate([rare[:2], [int(np.argmax(df))]]).astype(np.uint32)]
    qv = O.synth_rows_f32(len(q), DIM, stream=1)
    qv /= np.linalg.norm(qv, axis=1, keepdims=True)
    return q, qv


@pytest.mark.parametrize("name", ["configs0", "zipf200k", "adversarial"])
def test_shards_add_up_to_the_unsharded_build_and_rank_like_it(oi, corpora, name):
    from openintel_b200 import sharding
    texts = corpora[name]
    N = len(texts)
    csr, vocab = _host(texts)
    rows = _rows(N)
    q, qv = _queries(csr, vocab, N)
    with oi.GpuIndex(n_docs=N, dim=DIM, max_k=K, max_batch=4) as whole:
        whole.load_embeddings(rows)
        assert whole.build_bm25_text(texts) == vocab
        whole.bm25_finalize()
        want_bm = whole.search_bm25(q, K)
        want_cos = whole.search_cosine(qv, K)
    for world in (1, 2, 3, 8):
        shards, vocabs = _shards(oi, texts, world, rows)
        try:
            _check_shards(shards, vocabs, csr, vocab)
            _finalize_global(shards, N)
            for want, got in ((want_bm, [ix.search_bm25(q, K) for ix in shards]),
                              (want_cos, [ix.search_cosine(qv, K) for ix in shards])):
                ids, sc = sharding.merge_lists_host([g[0] for g in got], [g[1] for g in got], K)
                assert np.array_equal(ids, want[0]), (name, world)
                assert np.array_equal(sc.view(np.uint32), want[1].view(np.uint32)), (name, world)
        finally:
            for ix in shards:
                ix.close()


# ---- errors and state ---------------------------------------------------------------------------------------------
def _raw_union(ix, blob, offs, n, outs=True):
    nt, nb = C.c_uint32(), C.c_uint64()
    return ix.L.oi_index_bm25_union_vocabulary(ix.h, blob, offs, n, C.byref(nt) if outs else None, C.byref(nb) if outs else None)


def _pack(terms):
    from openintel_b200 import capi
    return capi.pack_texts(terms)


def _state(ix):
    b, o = ix.read_vocabulary_packed()
    _, _, npost = ix.bm25_local_stats()
    return [b.copy(), o.copy()] + list(_read_csr(ix, npost).values())


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def test_union_needs_an_unfinalized_part_built_from_text(oi):
    texts = ["alpha beta", "beta gamma", "gamma"]
    csr, vocab = _host(texts)
    blob, offs = _pack(vocab + ["delta"])
    with oi.GpuIndex(n_docs=3, dim=DIM, max_k=K) as ix:
        ix.load_embeddings(_rows(3))
        assert _raw_union(ix, blob.ctypes.data, offs.ctypes.data, len(offs) - 1) == 5  # no BM25 part at all
        ix.load_bm25(csr["term_offsets"], csr["doc_ids"], csr["tfs"], csr["doc_len"])
        assert _raw_union(ix, blob.ctypes.data, offs.ctypes.data, len(offs) - 1) == 5
        ix.synth_bm25(O.SEED, 50, O.zipf_cdf(50))
        assert _raw_union(ix, blob.ctypes.data, offs.ctypes.data, len(offs) - 1) == 5
        ix.build_bm25_text(texts)
        ix.bm25_finalize()
        with pytest.raises(oi.OiError) as e:
            ix.bm25_union_vocabulary(blob, offs)
        assert e.value.status == 5 and "finalized" in e.value.message


def test_bad_entries_leave_the_part_as_it_was(oi):
    texts = ["alpha beta zeta", "beta gamma", "gamma alpha0"]
    csr, vocab = _host(texts)
    assert vocab == ["alpha", "alpha0", "beta", "gamma", "zeta"]
    with oi.GpuIndex(n_docs=3, dim=DIM, max_k=K, max_batch=2) as ix:
        ix.load_embeddings(_rows(3))
        ix.build_bm25_text(texts)
        before = _state(ix)
        launches = ix.launch_count()

        def refused(blob, offs, n=None, status=1, outs=True, words=()):
            if n is None:
                n = len(offs) - 1
            assert _raw_union(ix, None if blob is None else blob.ctypes.data, None if offs is None else offs.ctypes.data,
                              n, outs) == status
            msg = ix.L.oi_last_error(ix.h).decode()
            for w in words:
                assert w in msg, msg
            assert _same(_state(ix), before)

        good = vocab + ["delta", "alpha"]
        blob, offs = _pack(good)
        refused(*_pack(["alpha", "alpha0", "beta", "delta", "zeta"]), words=("gamma", "missing"))  # a local term absent
        refused(*_pack(["alpha", "alpha0", "", "beta", "gamma", "zeta"]), words=("entry 2",))  # empty entry
        refused(*_pack(vocab + ["Alpha"]), words=("entry 5",))
        refused(*_pack(vocab[:2] + [b"del\x80ta"] + vocab[2:]), words=("entry 2",))
        bad = offs.copy()
        bad[3] = bad[2] - 1
        refused(blob, bad, words=("decrease",))
        refused(None, offs)
        refused(blob, None, n=len(offs) - 1)
        refused(blob, offs, outs=False)
        refused(blob, offs, n=0)
        assert ix.launch_count() > launches

        # a valid call afterwards succeeds, and is harmless when repeated, shuffled or duplicated
        g = sorted(set(good))
        assert ix.bm25_union_vocabulary(blob, offs) == g
        first = _state(ix)
        assert len(first[2]) == len(g) + 1 and first[2][g.index("delta") + 1] == first[2][g.index("delta")]
        assert ix.bm25_union_vocabulary(blob, offs) == g
        assert _same(_state(ix), first)
        rng = np.random.default_rng(3)
        shuffled = [good[i] for i in rng.permutation(len(good))] * 3
        assert ix.bm25_union_vocabulary(*_pack(shuffled)) == g
        assert _same(_state(ix), first)
        # the re-indexed part finalizes and searches like the host CSR over the same vocabulary
        ix.bm25_finalize()
        off = np.zeros(len(g) + 1, dtype=np.uint64)
        lens = np.zeros(len(g), dtype=np.uint64)
        lens[[g.index(w) for w in vocab]] = np.diff(csr["term_offsets"])
        off[1:] = np.cumsum(lens)
        with oi.GpuIndex(n_docs=3, dim=DIM, max_k=K, max_batch=2) as hx:
            hx.load_embeddings(_rows(3))
            hx.load_bm25(off, csr["doc_ids"], csr["tfs"], csr["doc_len"])
            hx.bm25_finalize()
            q = [np.array([g.index("alpha"), g.index("delta")], np.uint32), np.array([g.index("gamma")], np.uint32)]
            for a, c in zip(ix.search_bm25(q, 3), hx.search_bm25(q, 3)):
                assert np.array_equal(a.view(np.uint32), c.view(np.uint32))


# ---- the device lift out of the SQLite store, over gloo (both ranks on device 0) -----------------------------------
N_POSTS = 1500


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _lift_worker(rank, world, port, path, q):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from openintel_b200 import store
        conn = store.open_store(path)
        host = store.lift_shard(conn, dist)
        dev = store.lift_shard_gpu(conn, dist, device="cpu", device_index=0, max_k=K, max_batch=2)
        conn.close()
        ix = dev.pop("index")
        _, _, npost = ix.bm25_local_stats()
        csr = _read_csr(ix, npost)
        ix.close()
        q.put((rank, host, dev, csr))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,tokenless", [(2, False), (3, False), (3, True)])
def test_device_lift_equals_the_host_lift(oi, tmp_path, world, tokenless):
    """the device lift of every rank equals store.lift_shard's: vocabulary, CSR, global df / avgdl, post ids.  With
    `tokenless`, the middle shard's posts hold no token at all: it contributes no vocabulary and lifts empty lists."""
    import torch.multiprocessing as mp
    from openintel_b200 import sharding, store
    path = str(tmp_path / "posts.db")
    posts, _ = O.synth_posts(N_POSTS, 700, O.SEED)
    if tokenless:
        base, n = sharding.shard_range(N_POSTS, world, 1)
        for i in range(base, base + n):
            posts[i]["text"] = ("!!!", "\u00ff\u00fe ???", "... \u2014 !!", "\U0001f680 $$")[i % 4]
    conn = store.open_store(path, dim=8)
    store.insert_posts(conn, posts, np.ones((N_POSTS, 8), np.float32))
    conn.close()

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_lift_worker, args=(r, world, port, path, q)) for r in range(world)]
    [p.start() for p in procs]
    res = sorted([q.get(timeout=300) for _ in procs], key=lambda t: t[0])
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    for rank, host, dev, csr in res:
        assert (dev["doc_base"], dev["n_local"], dev["n_docs_global"]) == (host["doc_base"], host["n_local"], host["n_docs_global"])
        assert dev["vocab"] == host["vocab"] and dev["post_ids"] == host["post_ids"]
        assert np.array_equal(dev["global_df"], host["global_df"]) and dev["avgdl"] == host["avgdl"]
        for f in ("term_offsets", "doc_ids", "tfs", "doc_len"):
            assert np.array_equal(csr[f], host["csr"][f].astype(csr[f].dtype)), (rank, f)
        if tokenless and rank == 1:
            assert not len(csr["doc_ids"]) and not csr["doc_len"].any() and len(dev["vocab"]) > 100


def test_a_store_without_any_token_is_refused_with_the_build_error(oi, tmp_path):
    from openintel_b200 import store
    posts, _ = O.synth_posts(20, 50, O.SEED)
    for i, p in enumerate(posts):
        p["text"] = ("!!!", "\u00ff\u00fe ???")[i % 2]
    conn = store.open_store(str(tmp_path / "posts.db"), dim=8)
    store.insert_posts(conn, posts, np.ones((20, 8), np.float32))
    with pytest.raises(oi.OiError) as e:
        store.lift_shard_gpu(conn, None)
    assert e.value.status == 1 and "no token" in e.value.message
    conn.close()
