"""GPU parity of every cosine kernel path against the CPU oracle (SPEC §2).

Each search runs on a named path (`run_path`), and the launch count shows that the path was taken.  The paths are
checked at every class of accepted row width, at the size edges, and under inputs that only a wrong kernel gets
wrong: all scores negative, every score tied, exact duplicates spread over the CTAs, the best documents at either
end or in the partial last tile, and doc ids at the top of the u32 range.  Also here: the hybrid call's overlap
modes at small sizes and the widest accepted row."""
import numpy as np
import pytest

import oracle as O
from gpu_util import assert_ranked_close

pytestmark = pytest.mark.gpu

F32_TOL, BF16_TOL = 1e-5, 2e-3
MAX_DIM = 24576        # OI_MAX_DIM
GEMM_CAP = 512         # candidate-list capacity of the tensor-core kernel: it takes k + 64 <= 512
N_BIG = 100_003        # >= 100k rows, so the GEMM's probe and threshold ladder run; 100_003 % 64 = 35: a partial last tile
MAXERR = {}            # (path, dtype) -> largest |gpu - oracle| seen

# Options of each path, applied to a fresh handle (cosine_gemm_force_2d only acts at a handle's first GEMM call).
PATH_OPTS = {
    "ldg": dict(cosine_variant=0, cosine_multi_query=0, cosine_gemm_min_batch=0),
    "bulk": dict(cosine_variant=1, cosine_multi_query=0, cosine_gemm_min_batch=0),
    "multi1": dict(cosine_multi_query=1, cosine_gemm_min_batch=0),
    "multi2": dict(cosine_multi_query=2, cosine_gemm_min_batch=0),
    "fallback": {},  # default options, on a bf16 batch the tensor-core kernel refuses
    "gemm": {},
    "gemm_single": dict(cosine_gemm_pair=0),
    "gemm_2d": dict(cosine_gemm_pair=0, cosine_gemm_force_2d=1),  # the pair kernel always reads the 3-D view
    "gemm_lite": dict(cosine_gemm_lite=1),
    "gemm_ring24": dict(cosine_gemm_pair_ring=24),
}
SCAN_PATHS = ("ldg", "bulk", "multi1", "multi2")
GEMM_PATHS = ("gemm", "gemm_single", "gemm_2d", "gemm_lite", "gemm_ring24")


@pytest.fixture(scope="module")
def oi():
    import openintel_b200
    openintel_b200.load_library()
    yield openintel_b200
    print("\nlargest |gpu - oracle| by path and dtype:")
    for (path, dt), v in sorted(MAXERR.items()):
        print("  %-12s %-5s %.3g" % (path, dt, v))


@pytest.fixture(scope="module")
def num_sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _bf16(rows):
    return rows.dtype == np.uint16


def _nv(rows):
    """16-byte vectors per row: what the scan dispatch picks its kernel from"""
    return rows.shape[1] * rows.itemsize // 16


def gemm_eligible(rows, k):
    dim = rows.shape[1]
    return _bf16(rows) and dim % 64 == 0 and dim <= 768 and 24 % (dim // 64) == 0 and k + 64 <= GEMM_CAP


def scan_paths(rows, nq):
    """the scan paths that exist at this width and batch (the others would silently run a different kernel)"""
    nv, out = _nv(rows), ["ldg"]
    if nv <= 256:
        out.append("bulk")
    if nq >= 2 and nv <= 96:
        out.append("multi1")
        if 4 * ((nv + 31) // 32) * (8 if _bf16(rows) else 4) <= 48:
            out.append("multi2")
    return out


def gemm_paths(rows, nq, k):
    if not gemm_eligible(rows, k) or nq < 4:
        return []
    nkb, out = rows.shape[1] // 64, ["gemm", "gemm_single", "gemm_2d"]
    if 12 % nkb == 0:
        out.append("gemm_lite")
    if nkb == 12 and ((nq + 127) // 128) % 2 == 0:
        out.append("gemm_ring24")
    return out


def all_paths(rows, nq, k):
    out = scan_paths(rows, nq) + gemm_paths(rows, nq, k)
    if _bf16(rows) and nq >= 4 and not gemm_eligible(rows, k):
        out.append("fallback")
    return out


def expected_launches(path, rows, nq, k, num_sms, opts):
    """Kernel launches of one search call on `path`, the unpack kernel included.

    Scan: one launch per query (ldg, and the generic kernel that variant 1 also runs past 256 vectors), one persistent
    launch for the whole batch (bulk), one per group of 4 queries (multi1, multi2).  GEMM: query prep, main pass and
    merge, plus the probe pass and its merge on shards with at least 8 tiles per CTA.  The count cannot tell apart:
    ldg and bulk at nq = 1 (2 launches each); multi1 and multi2; the GEMM variants (pair, single CTA, 2-D view, lite
    ring, 24-slab pair ring), which differ only in the kernel launched.  `run_path` refuses the combinations in which a
    path would silently become another, so what the count cannot show is fixed by the arguments."""
    n, nv = len(rows), _nv(rows)
    if path in GEMM_PATHS:
        n_qt = (nq + 127) // 128
        pair = path in ("gemm", "gemm_ring24") and n_qt % 2 == 0
        ctas = num_sms & ~1 if pair else num_sms
        n_tiles = (n + 63) // 64
        n_ranges = min(max(1, ctas // n_qt), n_tiles)
        probe = opts.get("cosine_gemm_sample_tiles", 0) > 0 or (n_tiles + n_ranges - 1) // n_ranges >= 8
        return 4 + 2 * probe
    if path == "fallback":
        variant, multi = 1, 2
    else:
        variant, multi = opts.get("cosine_variant", 1), opts["cosine_multi_query"]
    if multi and nq >= 2 and nv <= 96:
        return (nq + 3) // 4 + 1
    if variant == 1 and nv <= 256:
        return 2
    return nq + 1


def run_path(oi, path, rows, qs, k, num_sms, doc_base=0, extra=None):
    """One search on a fresh handle on the named path; asserts the path applies and was taken -> (ids, scores, launches)"""
    n, dim = rows.shape
    nq = len(qs)
    if path == "fallback":
        assert _bf16(rows) and nq >= 4 and not gemm_eligible(rows, k)
    elif path in GEMM_PATHS:
        assert path in gemm_paths(rows, nq, k), (path, dim, nq, k)
    else:
        assert path in scan_paths(rows, nq), (path, dim, nq)
    opts = dict(PATH_OPTS[path], **(extra or {}))
    with oi.GpuIndex(n_docs=n, dim=dim, dtype=oi.DTYPE_BF16 if _bf16(rows) else oi.DTYPE_F32, max_k=k, max_batch=nq,
                     doc_base=doc_base) as ix:
        ix.load_embeddings(rows)
        for name, v in opts.items():
            ix.set_option(name, v)
        l0 = ix.launch_count()
        ids, sc = ix.search_cosine(qs, k)
        launches = ix.launch_count() - l0
    want = expected_launches(path, rows, nq, k, num_sms, opts)
    assert launches == want, "%s: %d launches, the path takes %d" % (path, launches, want)
    return ids, sc, launches


def oracle_scores(rows, qs):
    f = O.cosine_scores_bf16 if _bf16(rows) else O.cosine_scores_f32
    return np.stack([f(rows, q) for q in qs])


def check_lists(path, ids, sc, rows, allsc, k, doc_base=0):
    """every list against the oracle inside the SPEC §2 tie band; slots past n hold (NO_DOC, +0.0)"""
    n = len(rows)
    kk = min(k, n)
    bf16 = _bf16(rows)
    worst = 0.0
    for j in range(len(allsc)):
        wi, ws, _ = O.topk_f64(allsc[j], kk, doc_base=doc_base)
        assert_ranked_close(ids[j][:kk], sc[j][:kk], wi, ws, allsc[j], BF16_TOL if bf16 else F32_TOL, doc_base=doc_base)
        assert np.all(ids[j][kk:] == O.NO_DOC) and np.all(sc[j][kk:].view(np.uint32) == 0)
        worst = max(worst, float(np.max(np.abs(sc[j][:kk] - ws))))
    key = (path, "bf16" if bf16 else "f32")
    MAXERR[key] = max(MAXERR.get(key, 0.0), worst)


def queries(nq, dim, n):
    if nq == 1:
        return O.synth_rows_f32(1, dim, stream=1)
    return np.concatenate([O.synth_rows_f32(nq - 1, dim, stream=1), O.synth_planted_queries(1, dim, n)[0]])


def rows_of(dtype_name, n, dim):
    return O.synth_rows_bf16(n, dim) if dtype_name == "bf16" else O.synth_rows_f32(n, dim)


def to_dtype(rows_f32, dtype_name):
    return O.f32_to_bf16(rows_f32) if dtype_name == "bf16" else np.ascontiguousarray(rows_f32, dtype=np.float32)


def unit(v):
    v = np.asarray(v, dtype=np.float64)
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


# ---- 2. row widths ----------------------------------------------------------------------------------------------
# f32: 516 and 772 are the padded NVL 5 -> 6 and 7 -> 8 cases, 1028 and up the generic kernel; bf16 likewise at
# 1032, 1544 and 2056.  320, 448, 640 and everything past 768 or off a multiple of 64 are bf16 widths the GEMM refuses.
F32_WIDTHS = [4, 12, 100, 128, 132, 384, 388, 516, 772, 1024, 1028, 3000, MAX_DIM]
BF16_WIDTHS = [8, 40, 200, 256, 264, 320, 448, 640, 768, 776, 1032, 1544, 2048, 2056, 4096, MAX_DIM]


@pytest.mark.parametrize("dtype_name,dim", [("f32", d) for d in F32_WIDTHS] + [("bf16", d) for d in BF16_WIDTHS])
def test_every_path_at_every_width(oi, num_sms, dtype_name, dim):
    """every path that exists at the width matches the oracle and the ldg kernel; MAX_DIM is the widest accepted row"""
    n = 20011 if dim <= 1024 else 5003 if dim <= 4096 else 3001
    k = 37
    rows = rows_of(dtype_name, n, dim)
    for nq in (1, 5, 130):
        paths = [p for p in all_paths(rows, nq, k) if nq != 130 or p in GEMM_PATHS]
        if not paths:
            continue
        qs = queries(nq, dim, n)
        allsc = oracle_scores(rows, qs)
        ref_ids, ref_sc, _ = run_path(oi, "ldg", rows, qs, k, num_sms)
        check_lists("ldg", ref_ids, ref_sc, rows, allsc, k)
        for path in paths:
            if path == "ldg":
                continue
            ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms)
            check_lists(path, ids, sc, rows, allsc, k)
            assert np.max(np.abs(sc - ref_sc)) <= 2e-6, (path, float(np.max(np.abs(sc - ref_sc))))


# ---- 3. size edges ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
@pytest.mark.parametrize("n", [1, 31, 63, 64, 65, 129])
def test_size_edges(oi, num_sms, dtype_name, n):
    dim = 128
    rows = rows_of(dtype_name, n, dim)
    for k in sorted({1, n, n + 7}):
        for nq in (1, 5, 130):
            qs = O.synth_rows_f32(nq, dim, stream=1)
            allsc = oracle_scores(rows, qs)
            for path in all_paths(rows, nq, k):
                if nq == 130 and path not in GEMM_PATHS:
                    continue
                ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms, doc_base=3)
                check_lists(path, ids, sc, rows, allsc, k, doc_base=3)


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
def test_max_k_on_every_scan_path(oi, num_sms, dtype_name):
    """k = 1024 over 100k rows: the final merge of the per-CTA lists is too large for its in-buffer branch"""
    k, dim = 1024, 128
    rows = rows_of(dtype_name, N_BIG, dim)
    for nq in (1, 5):
        qs = queries(nq, dim, N_BIG)
        allsc = oracle_scores(rows, qs)
        for path in scan_paths(rows, nq):
            ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms)
            check_lists(path, ids, sc, rows, allsc, k)


@pytest.mark.parametrize("k", [448, 449, 1024])
def test_bf16_batch_either_side_of_the_gemm_k_bound(oi, num_sms, k):
    """default options: k + 64 <= 512 takes the tensor cores, a larger k falls back to the scan"""
    dim, nq = 128, 5
    rows = O.synth_rows_bf16(N_BIG, dim)
    qs = queries(nq, dim, N_BIG)
    path = "gemm" if k + 64 <= GEMM_CAP else "fallback"
    ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms)
    check_lists(path, ids, sc, rows, oracle_scores(rows, qs), k)


# ---- 4. adversarial score distributions -------------------------------------------------------------------------
def _big_paths(rows, nq, k):
    return scan_paths(rows, nq) + gemm_paths(rows, nq, k)


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
def test_all_scores_negative(oi, num_sms, dtype_name):
    """Rows in a half-space (synthetic rows pushed along u, renormalised) and queries near -u: every score is
    negative, so the zero-filled columns of the GEMM's partial last tile would outrank every document if they were
    let in.  k = 4: the partial tile holds 4 groups of 8 columns with a zero column, so a probe that sampled it would
    put its first rung at 0 and reject every document.  cosine_gemm_sample_tiles = 56 makes the probe cover every tile."""
    dim, doc_base = 128, 1000
    u = unit(O.synth_rows_f32(1, dim, stream=2)[0])
    rows = to_dtype(unit(O.synth_rows_f32(N_BIG, dim).astype(np.float64) + 2.0 * u), dtype_name)
    w = O.synth_rows_f32(4, dim, stream=1).astype(np.float64)
    qs = np.concatenate([-u[None], unit(-u + 0.3 * w)]).astype(np.float32)
    allsc = oracle_scores(rows, qs)
    assert allsc.max() < -0.1
    for k in (4, 100):
        for path in _big_paths(rows, len(qs), k):
            for extra in ([None, dict(cosine_gemm_sample_tiles=56)] if path == "gemm" else [None]):
                ids, sc, launches = run_path(oi, path, rows, qs, k, num_sms, doc_base=doc_base, extra=extra)
                if path in GEMM_PATHS:
                    assert launches == 6  # the probe ran
                assert np.all(ids < doc_base + N_BIG), (path, extra)
                check_lists(path, ids, sc, rows, allsc, k, doc_base=doc_base)


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
@pytest.mark.parametrize("zero", [0.0, -0.0])
def test_zero_query_ties_every_document(oi, num_sms, dtype_name, zero):
    """every score is 0: every document passes every threshold, and the doc id alone decides the order"""
    dim, doc_base = 128, 77
    rows = rows_of(dtype_name, N_BIG, dim)
    qs = np.full((5, dim), zero, dtype=np.float32)
    for k in (10, 448, 1024):
        for path in _big_paths(rows, len(qs), k):
            ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms, doc_base=doc_base)
            assert np.array_equal(ids, np.tile(np.arange(doc_base, doc_base + k, dtype=np.uint32), (len(qs), 1))), path
            assert np.all(sc.view(np.uint32) == 0), path  # +0.0, never -0.0


def _separated_rows(dim, m):
    """m unit rows whose scores against qhat are spread evenly over [-0.9, 0.9] -> (rows f64, qhat)"""
    qhat = unit(O.synth_rows_f32(1, dim, stream=3)[0])
    v = O.synth_rows_f32(m, dim, stream=4).astype(np.float64)
    v = unit(v - np.outer(v @ qhat, qhat))
    c = np.random.default_rng(5).permutation(np.linspace(-0.9, 0.9, m))
    return c[:, None] * qhat + np.sqrt(1 - c * c)[:, None] * v, qhat


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
def test_exact_duplicates_across_ctas(oi, num_sms, dtype_name):
    """256 distinct rows, each repeated ~390 times in a shuffled order over 100k rows: the k-th score is shared by
    hundreds of documents in different CTAs.  Identical rows must score bit-identically on every path, so the
    expected list is exact (score descending, then doc id) and the GPU ids must equal it position by position."""
    dim, m, doc_base = 128, 256, 9
    tol = BF16_TOL if dtype_name == "bf16" else F32_TOL
    distinct, qhat = _separated_rows(dim, m)
    distinct = to_dtype(distinct, dtype_name)
    for nq in (5, 130):
        w = O.synth_rows_f32(nq, dim, stream=1).astype(np.float64)
        sign = np.where(np.arange(nq) % 2 == 0, 1.0, -1.0)[:, None]
        qs = unit(sign * qhat + 0.01 * w).astype(np.float32)
        dsc = oracle_scores(distinct, qs)
        gaps = np.diff(np.sort(dsc, axis=1), axis=1)
        assert np.all(gaps > tol * np.maximum(np.abs(dsc).max(axis=1, keepdims=True), 1e-2))
        src = np.random.default_rng(7).permutation(np.resize(np.arange(m), N_BIG))
        rows = np.ascontiguousarray(distinct[src])
        allsc = dsc[:, src]
        docs = np.arange(N_BIG)
        exact = np.stack([np.lexsort((docs, -allsc[j]))[:1024] + doc_base for j in range(nq)]).astype(np.uint32)
        for k in (100, 448, 1024):
            want = exact[:, :k]
            for path in _big_paths(rows, nq, k):
                if nq == 130 and path not in GEMM_PATHS:
                    continue
                ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms, doc_base=doc_base)
                assert np.array_equal(ids, want), (path, nq, k, int(np.sum(ids != want)))
                check_lists(path, ids, sc, rows, allsc, k, doc_base=doc_base)


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
@pytest.mark.parametrize("order", ["ascending", "descending", "last_tile"])
def test_order_of_the_best_documents(oi, num_sms, dtype_name, order):
    """for the first query: scores ascending with the doc id (every tile raises the threshold), descending (the
    first tiles settle it), or the best k all in the partial last tile"""
    dim, k = 128, 32
    rows = rows_of(dtype_name, N_BIG, dim)
    qs = queries(5, dim, N_BIG)
    s0 = oracle_scores(rows, qs[:1])[0]
    if order == "ascending":
        perm = np.argsort(s0, kind="stable")
    elif order == "descending":
        perm = np.argsort(-s0, kind="stable")
    else:
        best = np.argsort(-s0, kind="stable")[:N_BIG % 64]
        perm = np.concatenate([np.setdiff1d(np.arange(N_BIG), best), best])
    rows = np.ascontiguousarray(rows[perm])
    allsc = oracle_scores(rows, qs)
    if order == "last_tile":
        assert np.all(O.topk_f64(allsc[0], k)[0] >= N_BIG - N_BIG % 64)
    for path in _big_paths(rows, len(qs), k):
        ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms)
        check_lists(path, ids, sc, rows, allsc, k)


@pytest.mark.parametrize("dtype_name", ["f32", "bf16"])
@pytest.mark.parametrize("n,k", [(129, 136), (N_BIG, 100)])
def test_doc_ids_at_the_top_of_the_u32_range(oi, num_sms, dtype_name, n, k):
    """doc_base + n = 2^32 - 2: the last doc id is 0xFFFFFFFD, two below the NO_DOC padding"""
    dim = 128
    doc_base = 2 ** 32 - 2 - n
    rows = rows_of(dtype_name, n, dim)
    qs = queries(5, dim, n)
    allsc = oracle_scores(rows, qs)
    for path in _big_paths(rows, len(qs), k):
        ids, sc, _ = run_path(oi, path, rows, qs, k, num_sms, doc_base=doc_base)
        assert np.all(ids[:, :min(k, n)] != O.NO_DOC) and np.all(ids[:, :min(k, n)] >= doc_base), path
        check_lists(path, ids, sc, rows, allsc, k, doc_base=doc_base)


# ---- 5. hybrid overlap modes ------------------------------------------------------------------------------------
def _bm25_oracle_lists(corp, qt, n, k):
    w = O.bm25_weights(corp["term_offsets"], corp["doc_ids"], corp["tfs"], corp["doc_len"],
                       O.bm25_idf(n, np.diff(corp["term_offsets"])))
    out = []
    for q in qt:
        s = O.bm25_score_dense(corp["term_offsets"], corp["doc_ids"], w, np.asarray(q, dtype=np.uint32), n)
        out.append(O.topk_f32(s, k, only_positive=True)[0])
    return out


@pytest.mark.parametrize("dim", [128, 768])
@pytest.mark.parametrize("mode,gemm_sms", [(1, 74), (2, 2), (2, 3), (2, 74)])
def test_hybrid_overlap_modes(oi, dim, mode, gemm_sms):
    """the hybrid call with its two legs overlapped (1: lite GEMM next to BM25 on every SM; 2: the GEMM on gemm_sms
    SMs) returns the RRF of the oracle-checked cosine list and the oracle BM25 list, bit for bit"""
    n, vocab, k = 20011, 2000, 20
    rows = O.synth_rows_bf16(n, dim)
    corp = O.synth_bm25_corpus(n, vocab)
    with oi.GpuIndex(n_docs=n, dim=dim, dtype=oi.DTYPE_BF16, max_k=k, max_batch=130) as ix:
        ix.load_embeddings(rows)
        ix.load_bm25(corp["term_offsets"], corp["doc_ids"], corp["tfs"], corp["doc_len"])
        ix.bm25_finalize()
        ix.set_option("hybrid_overlap", mode)
        ix.set_option("overlap_gemm_sms", gemm_sms)
        for nq in (6, 130):
            qs = queries(nq, dim, n)
            qt = O.synth_query_terms(nq, 8, corp["cdf"])
            cos_ids, cos_sc = ix.search_cosine(qs, k)
            check_lists("hybrid_cos", cos_ids, cos_sc, rows, oracle_scores(rows, qs), k)
            bm_ids = _bm25_oracle_lists(corp, qt, n, k)
            ids, rrf, rc, rb = ix.search_hybrid(qs, qt, k)
            for j in range(nq):
                e_ids, e_val, e_rc, e_rb, _ = O.rrf(cos_ids[j], bm_ids[j], k)
                assert np.array_equal(ids[j], e_ids) and np.array_equal(rrf[j].view(np.uint32), e_val.view(np.uint32))
                assert np.array_equal(rc[j], e_rc) and np.array_equal(rb[j], e_rb)


# ---- 6. the dim limit -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype_name,dim", [("f32", MAX_DIM + 4), ("bf16", MAX_DIM + 8)])
def test_dim_past_the_limit_is_refused_at_create(oi, dtype_name, dim):
    """the next width past MAX_DIM is refused at create: no cosine kernel could search it (MAX_DIM itself is
    searched in test_every_path_at_every_width)"""
    with pytest.raises(oi.OiError) as e:
        oi.GpuIndex(n_docs=100, dim=dim, dtype=oi.DTYPE_BF16 if dtype_name == "bf16" else oi.DTYPE_F32)
    assert e.value.status == 1 and str(MAX_DIM) in e.value.message
