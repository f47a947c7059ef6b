"""Host-side plumbing of the document-sharded index (docs/SPEC.md §5): one process per GPU,
contiguous doc ranges, GLOBAL BM25 statistics, and the NCCL communicator the C library uses for
the all-gather of local top-k lists.  torch.distributed is used only as the control plane
(all-gather of the shards' vocabularies and all-reduce of df / doc-length sums at build time,
broadcast of the NCCL unique id); the
per-query exchange itself is libopenintel_gpu.so's ncclAllGather + device merge.

The same functions run over gloo on CPU tensors (tests/test_sharding_gloo.py) and over NCCL.
"""
import numpy as np

from . import capi


def shard_range(n_docs, world, rank):
    """SPEC §5: shard r of G holds [r*ceil(N/G), min(N, (r+1)*ceil(N/G))).  -> (doc_base, n_local)"""
    if world < 1 or not 0 <= rank < world:
        raise ValueError("rank %d / world %d" % (rank, world))
    per = (n_docs + world - 1) // world
    base = min(n_docs, rank * per)
    return base, max(0, min(n_docs, base + per) - base)


def global_bm25_stats(dist, df_local, sum_doc_len_local, n_docs_local, device="cpu"):
    """All-reduce the shard statistics into the GLOBAL (df[n_terms] u32, avgdl f32, N) every shard
    must score with, so that a sharded index ranks exactly like an unsharded one (SPEC §3/§5).
    `dist` is torch.distributed (initialised) or None for a single shard."""
    df = np.ascontiguousarray(df_local, dtype=np.uint32)
    if dist is None or dist.get_world_size() == 1:
        n = int(n_docs_local)
        return df, np.float32(np.float64(sum_doc_len_local) / n) if n else np.float32(1.0), n
    import torch
    t_df = torch.from_numpy(df.astype(np.int64)).to(device)
    t_sc = torch.tensor([int(sum_doc_len_local), int(n_docs_local)], dtype=torch.int64, device=device)
    dist.all_reduce(t_df, op=dist.ReduceOp.SUM)
    dist.all_reduce(t_sc, op=dist.ReduceOp.SUM)
    gdf = t_df.cpu().numpy()
    if gdf.max(initial=0) > 0xFFFFFFFF:
        raise OverflowError("global df does not fit u32")
    s, n = (int(x) for x in t_sc.cpu().tolist())
    avgdl = np.float32(np.float64(s) / np.float64(n)) if n else np.float32(1.0)
    return gdf.astype(np.uint32), avgdl, n


def all_gather_packed(dist, blob, offsets, device="cpu"):
    """Every rank's byte strings, packed as (blob u8[], offsets u64[n + 1]: string i = blob[offsets[i] .. offsets[i + 1]))
    -> all ranks' strings concatenated in rank order, packed the same way (offsets from 0).  Used to gather the shards'
    vocabularies for oi_index_bm25_union_vocabulary without decoding them to Python strings.  `dist` is
    torch.distributed (initialised) or None for a single shard."""
    blob = np.ascontiguousarray(blob, dtype=np.uint8)
    offs = np.ascontiguousarray(offsets, dtype=np.int64)
    mine, lens = blob[offs[0]:offs[-1]], np.diff(offs)
    if dist is None or dist.get_world_size() == 1:
        return mine.copy(), np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    import torch
    world = dist.get_world_size()
    size = torch.tensor([len(mine), len(lens)], dtype=torch.int64, device=device)
    sizes = [torch.zeros_like(size) for _ in range(world)]
    dist.all_gather(sizes, size)
    sizes = [tuple(int(x) for x in t.cpu().tolist()) for t in sizes]
    # padded to the largest rank's share, at least one element (a rank may hold nothing)
    nb, nl = max(max(s[0] for s in sizes), 1), max(max(s[1] for s in sizes), 1)
    t_blob = torch.zeros(nb, dtype=torch.uint8)
    t_blob[:len(mine)] = torch.from_numpy(mine)
    t_lens = torch.zeros(nl, dtype=torch.int64)
    t_lens[:len(lens)] = torch.from_numpy(lens)
    t_blob, t_lens = t_blob.to(device), t_lens.to(device)
    g_blob = [torch.empty_like(t_blob) for _ in range(world)]
    g_lens = [torch.empty_like(t_lens) for _ in range(world)]
    dist.all_gather(g_blob, t_blob)
    dist.all_gather(g_lens, t_lens)
    out_blob = np.concatenate([g.cpu().numpy()[:s[0]] for g, s in zip(g_blob, sizes)])
    out_lens = np.concatenate([g.cpu().numpy()[:s[1]] for g, s in zip(g_lens, sizes)])
    return out_blob, np.concatenate([[0], np.cumsum(out_lens)]).astype(np.uint64)


def _relay_states(dist, n, run, device="cpu"):
    """The relay of n running states over the ranks in rank order (SPEC §8a): rank 0 runs `run(None)`, every later rank
    receives the states of rank - 1 and runs `run(carry)`, and sends its states on; the last rank broadcasts its states
    and summaries.  run(carry) -> (states: MENTION_STATE_DTYPE [n], summaries: SOCIAL_SUMMARY_DTYPE [n]).
    -> the last rank's (states, summaries) on every rank."""
    import torch
    rank, world = dist.get_rank(), dist.get_world_size()
    carry = None
    if rank > 0:
        buf = torch.empty(n * capi.MENTION_STATE_DTYPE.itemsize, dtype=torch.uint8, device=device)
        dist.recv(buf, src=rank - 1)
        carry = buf.cpu().numpy().view(capi.MENTION_STATE_DTYPE)
    states, raw = run(carry)
    states = np.ascontiguousarray(states).reshape(-1)
    if rank < world - 1:
        dist.send(torch.from_numpy(states.view(np.uint8).copy()).to(device), dst=rank + 1)
    # the last rank's states and summaries, as bytes, to everybody
    raw = np.ascontiguousarray(raw).reshape(-1) if rank == world - 1 else np.zeros(n, dtype=capi.SOCIAL_SUMMARY_DTYPE)
    out = torch.from_numpy(np.concatenate([states.view(np.uint8), raw.view(np.uint8)])).to(device)
    dist.broadcast(out, world - 1)
    out = out.cpu().numpy()
    cut = n * capi.MENTION_STATE_DTYPE.itemsize
    return out[:cut].copy().view(capi.MENTION_STATE_DTYPE), out[cut:].copy().view(capi.SOCIAL_SUMMARY_DTYPE)


def relay_mention_summary(dist, ix, term_ids, source=None, threshold=0.2, device="cpu"):
    """The social summaries of `term_ids` over the posting lists of a document-sharded index (SPEC §8a), the same on
    every rank: rank 0 summarises its shard and sends its running states to rank 1; every later rank receives them,
    continues each term's chain over its own shard (GpuIndex.mention_summary with carry) and sends on; the last rank
    broadcasts the final states and summaries.

    The relay is sequential over the ranks by design: the reference's mean is a sequential f64 sum in doc order and the
    shards hold contiguous doc ranges in rank order, so only carrying the running sum from shard to shard reproduces it
    bit for bit -- an all-reduce of per-shard partial sums would round differently.  `dist` = torch.distributed
    (initialised) or None for a single shard; every rank passes the same term ids.  -> (states, summaries) as
    GpuIndex.mention_summary returns them."""
    if dist is None or dist.get_world_size() == 1 or len(term_ids) == 0:
        return ix.mention_summary(term_ids, source, threshold)

    def run(carry):
        states, sums = ix.mention_summary(term_ids, source, threshold, carry)
        return states, capi.summaries_to_array(sums)
    states, raw = _relay_states(dist, len(term_ids), run, device)
    return states, capi.summaries_from_array(raw)


def relay_mention_timeline(dist, ix, term_ids, edges, source=None, threshold=0.2, device="cpu"):
    """The per-(term, bucket) summaries of a document-sharded index (SPEC §8b), the same on every rank: the relay of
    relay_mention_summary over the n x B running states of GpuIndex.mention_timeline.  Every rank passes the same term
    ids and edges.  -> (states [n][B], summaries: n lists of B dicts) as GpuIndex.mention_timeline returns them."""
    if dist is None or dist.get_world_size() == 1 or len(term_ids) == 0:
        return ix.mention_timeline(term_ids, edges, source, threshold)
    n, nb = len(term_ids), len(edges) - 1

    def run(carry):
        states, sums = ix.mention_timeline(term_ids, edges, source, threshold,
                                           None if carry is None else carry.reshape(n, nb))
        return states, capi.summaries_to_array([sm for row in sums for sm in row])
    states, raw = _relay_states(dist, n * nb, run, device)
    sums = capi.summaries_from_array(raw)
    return states.reshape(n, nb), [sums[i * nb:(i + 1) * nb] for i in range(n)]


def all_reduce_counts(dist, counts, device="cpu"):
    """The global mention counts of a document-sharded index (SPEC §8c): the sum of the shards' counts, the same on
    every rank.  Integers, so an all-reduce is exact in any order and no relay is needed; the shards' arrays line up
    because the vocabulary is the global union (SPEC §5).  `dist` = torch.distributed (initialised) or None for a single
    shard.  -> int64 array shaped like `counts`"""
    out = np.asarray(counts).astype(np.int64)
    if dist is None or dist.get_world_size() == 1:
        return out
    import torch
    t = torch.from_numpy(out).to(device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t.cpu().numpy()


def relay_comention_summary(dist, ix, anchor_ids, term_ids, window, source=None, threshold=0.2, device="cpu"):
    """The shared-post summaries of the pairs (anchor_ids[j], term_ids[j]) over a document-sharded index (SPEC §8d), the
    same on every rank: the relay of relay_mention_summary over the states of GpuIndex.comention_summary.  The post
    masks are shard-local; only the states cross ranks.  Every rank passes the same pairs and window.  -> (states,
    summaries) as GpuIndex.comention_summary returns them."""
    if dist is None or dist.get_world_size() == 1 or len(term_ids) == 0:
        return ix.comention_summary(anchor_ids, term_ids, window, source, threshold)

    def run(carry):
        states, sums = ix.comention_summary(anchor_ids, term_ids, window, source, threshold, carry)
        return states, capi.summaries_to_array(sums)
    states, raw = _relay_states(dist, len(term_ids), run, device)
    return states, capi.summaries_from_array(raw)


def all_gather_runs(dist, runs, device="cpu"):
    """Every rank's author runs (capi.AUTHOR_RUN_DTYPE, any number per rank) -> the list of all ranks' runs in rank
    order, the same on every rank (SPEC §8e), as the bytes of all_gather_packed.  `dist` = torch.distributed
    (initialised) or None for a single shard."""
    raw = np.ascontiguousarray(runs, dtype=capi.AUTHOR_RUN_DTYPE).view(np.uint8)
    blob, offs = all_gather_packed(dist, raw, np.array([0, len(raw)]), device=device)
    offs = offs.astype(np.int64)
    return [blob[offs[r]:offs[r + 1]].copy().view(capi.AUTHOR_RUN_DTYPE) for r in range(len(offs) - 1)]


def broadcast_unique_id(dist, device="cpu"):
    """rank 0 creates the NCCL unique id (C ABI), everybody receives it."""
    import torch
    uid = torch.zeros(capi.UNIQUE_ID_BYTES, dtype=torch.uint8)
    if dist.get_rank() == 0:
        uid = torch.from_numpy(capi.GpuIndex.comm_unique_id().copy())
    uid = uid.to(device)
    dist.broadcast(uid, 0)
    return uid.cpu().numpy()


def attach_p2p(dist, ix, device="cpu"):
    """Switch a shard's exchange from ncclAllGather to the peer-to-peer push (all ranks on one NVLink box): every rank
    exports the IPC handle of its exchange buffer, the handles are all-gathered through torch.distributed (control
    plane), every rank maps its peers' buffers."""
    import torch
    mine = torch.from_numpy(ix.p2p_export().copy()).to(device)
    allh = [torch.zeros_like(mine) for _ in range(dist.get_world_size())]
    dist.all_gather(allh, mine)
    ix.p2p_attach(np.stack([t.cpu().numpy() for t in allh]))


def merge_lists_host(ids_per_rank, scores_per_rank, k):
    """Reference model of the device merge for tests: G lists [nq][k] -> best k by SPEC §1 order
    (score desc, doc id asc; NO_DOC padding dropped).  Not used by the product path."""
    ids = np.concatenate(ids_per_rank, axis=1).astype(np.uint32)
    sc = np.concatenate(scores_per_rank, axis=1).astype(np.float32)
    nq = ids.shape[0]
    out_ids = np.full((nq, k), capi.NO_DOC, dtype=np.uint32)
    out_sc = np.zeros((nq, k), dtype=np.float32)
    for j in range(nq):
        keep = ids[j] != capi.NO_DOC
        i, s = ids[j][keep], sc[j][keep] + np.float32(0.0)
        order = np.lexsort((i, -s.astype(np.float64)))[:k]
        out_ids[j, :len(order)] = i[order]
        out_sc[j, :len(order)] = s[order]
    return out_ids, out_sc


class ShardedIndex:
    """One rank's shard of a doc-sharded hybrid index.  Builds the shard (synthetic, SPEC §9, or
    from caller-provided arrays), agrees on global BM25 statistics and wires the communicator."""

    def __init__(self, n_docs_global, dim, dtype=capi.DTYPE_F32, dist=None, device_index=0, max_k=100, max_batch=1, exchange="nccl"):
        self.dist = dist if (dist is not None and dist.get_world_size() > 1) else None
        self.rank = self.dist.get_rank() if self.dist else 0
        self.world = self.dist.get_world_size() if self.dist else 1
        self.n_docs_global = int(n_docs_global)
        self.doc_base, self.n_local = shard_range(self.n_docs_global, self.world, self.rank)
        self.device_index = device_index
        self.ix = capi.GpuIndex(n_docs=self.n_local, dim=dim, dtype=dtype, device=device_index, doc_base=self.doc_base,
                                max_k=max_k, max_batch=max_batch)
        if self.dist:
            uid = broadcast_unique_id(self.dist, device="cuda:%d" % device_index)
            self.ix.comm_init(self.rank, self.world, uid)
            if exchange == "p2p":
                attach_p2p(self.dist, self.ix, device="cuda:%d" % device_index)

    def synth(self, seed, vocab=None, zipf_cdf=None, k1=1.2, b=0.75):
        self.ix.synth_embeddings(seed)
        if vocab:
            self.ix.synth_bm25(seed, vocab, zipf_cdf)
            self.finalize_bm25(k1, b)
        return self

    def finalize_bm25(self, k1=1.2, b=0.75):
        df, sdl, _ = self.ix.bm25_local_stats()
        gdf, avgdl, n = global_bm25_stats(self.dist, df, sdl, self.n_local, device="cuda:%d" % self.device_index)
        assert n == self.n_docs_global
        self.global_df, self.avgdl = gdf, avgdl
        self.ix.bm25_finalize(k1=k1, b=b, avgdl=float(avgdl), n_docs_global=n, global_df=gdf)

    def close(self):
        self.ix.close()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()
